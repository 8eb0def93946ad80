"""Mixed-map environments on the GPU: every map's slice of one mixed environment is, bit for bit, the single-map
environment of that map with gid0 + its offset — state, records and the learner layouts — across list / rasteriser
sensors, the specialised / any-shape kernels, one-wave / persistent launches and a grid capped below the map count;
and every other entry point (masked reset, observe, state access, the host-buffer path, graph capture, the learner and
the evaluator) works on one."""
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import selfplay
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import load_named_map
from as_cops_and_thieves_b200.worlds import CatWorlds

pytestmark = pytest.mark.gpu

NAMES = ("squarinth", "agh-map", "labyrinth")
SHAPES = {"one_wave": (1, 37, 4096), "persistent": (1, 37, 12000), "max_grid": (1, 37, 4096)}


def _pair(cuda_device, counts, seed=5, gid0=11, **kw):
    """A mixed environment of NAMES with `counts` worlds and the single-map environments of its slices."""
    cmaps = [pu.named_cmap(n) for n in NAMES]
    mixed = CatWorlds(cmaps, counts, device=cuda_device, gid0=gid0, seed=seed, **kw)
    singles = [CatWorlds(c, n, device=cuda_device, gid0=gid0 + off, seed=seed, **kw)
               for c, n, off in zip(cmaps, counts, mixed.world_offsets)]
    return mixed, singles


def _slices(mixed):
    return [slice(o, o + n) for o, n in zip(mixed.world_offsets, mixed.worlds_per_map)]


def _assert_same(mixed, singles, what):
    N = mixed.n_worlds
    st = mixed.state.view(N, -1)
    rec = mixed._out.view(N, -1)
    for s, w in zip(_slices(mixed), singles):
        assert torch.equal(st[s], w.state.view(w.n_worlds, -1)), f"{what}: state"
        assert torch.equal(rec[s], w._out.view(w.n_worlds, -1)), f"{what}: records"
        for name in ("obs_f32", "state_f32", "critic_f32"):
            a, b = getattr(mixed, name), getattr(w, name)
            if a is None:
                continue
            a = a[:, s] if name == "obs_f32" else a[s]
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{what}: {name}"


@pytest.mark.parametrize("sensor", ["lists", "raster"])
@pytest.mark.parametrize("kernel", ["shipped", "generic", "rays37"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_slices_equal_single_map_environments(cuda_device, monkeypatch, sensor, kernel, shape):
    if kernel == "generic" and shape == "persistent":
        pytest.skip("the any-shape kernel's persistent launches are covered by rays37")
    kw = dict(want_critic=True, max_step_count=60)
    if sensor == "raster":
        kw["ray_list_cell"] = -1.0
    if kernel == "generic":
        monkeypatch.setenv("CAT_GENERIC_KERNEL", "1")
    if kernel == "rays37":
        kw["n_rays"] = 37
    if shape == "max_grid":
        monkeypatch.setenv("CAT_MAX_GRID", "2")
    counts = SHAPES[shape]
    mixed, singles = _pair(cuda_device, counts, **kw)
    monkeypatch.delenv("CAT_GENERIC_KERNEL", raising=False)
    monkeypatch.delenv("CAT_MAX_GRID", raising=False)
    if shape == "max_grid":
        assert mixed.info.grid == len(NAMES)                        # raised to one CTA per map
    N = mixed.n_worlds
    assert mixed.info.n_worlds == N and mixed.info.map_blob_bytes == max(mixed.map_info(m).map_blob_bytes for m in range(3))
    assert mixed.info.ray_list_bytes == sum(mixed.map_info(m).ray_list_bytes for m in range(3))
    for m, w in enumerate(singles):
        mi = mixed.map_info(m)
        assert mi.n_worlds == counts[m] and mi.n_edges == w.info.n_edges and mi.ray_list_bytes == w.info.ray_list_bytes
    assert torch.equal(mixed.map_index.cpu(), torch.repeat_interleave(torch.arange(3), torch.tensor(counts)))
    mixed.reset()
    for w in singles:
        w.reset()
    _assert_same(mixed, singles, "reset")
    g = torch.Generator().manual_seed(7)
    done = 0
    for t in range(200):
        a = torch.randint(0, 4, (N, mixed.A), dtype=torch.uint8, generator=g).to(cuda_device)
        mixed.step(a)
        for s, w in zip(_slices(mixed), singles):
            w.step(a[s].contiguous())
        _assert_same(mixed, singles, f"step {t}")
        done += int(mixed.terminated.sum())
    assert done > 0, "no world finished: the auto-reset path was not exercised"
    assert mixed.overflow_counts() == (0, 0)
    mixed.close()
    for w in singles:
        w.close()


def test_masked_reset_observe_and_state_round_trip(cuda_device):
    counts = (1, 37, 4096)
    mixed, singles = _pair(cuda_device, counts, want_critic=True, max_step_count=60)
    N = mixed.n_worlds
    mixed.reset()
    for w in singles:
        w.reset()
    g = torch.Generator().manual_seed(3)
    for _ in range(10):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
        mixed.step(a)
        for s, w in zip(_slices(mixed), singles):
            w.step(a[s].contiguous())
    mask = (torch.rand(N, generator=g) < 0.3).to(torch.uint8)
    mask[0] = 1
    mixed.reset(mask)
    for s, w in zip(_slices(mixed), singles):
        w.reset(mask[s])
    _assert_same(mixed, singles, "masked reset")
    mixed.observe()
    for w in singles:
        w.observe()
    _assert_same(mixed, singles, "observe")
    # get_state of the mixed environment = the slices' get_state; set_state of it, then a step, stays equal
    st = mixed.get_state()
    for s, w in zip(_slices(mixed), singles):
        ws = w.get_state()
        for k in st:
            assert torch.equal(st[k][s], ws[k]), k
    st["pos"] += 0.25
    mixed.set_state(pos=st["pos"])
    for s, w in zip(_slices(mixed), singles):
        w.set_state(pos=st["pos"][s])
    a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
    mixed.step(a)
    for s, w in zip(_slices(mixed), singles):
        w.step(a[s].contiguous())
    _assert_same(mixed, singles, "step after set_state")


@pytest.mark.parametrize("packed", [True, False], ids=["packed", "u8"])
def test_step_host_modes_match_device_records(cuda_device, packed):
    counts = (1, 37, 4096)
    cmaps = [pu.named_cmap(n) for n in NAMES]
    kw = dict(device=cuda_device, seed=9, want_f32=False, want_shared=False, max_step_count=50)
    dev_env, host_env = CatWorlds(cmaps, counts, **kw), CatWorlds(cmaps, counts, **kw)
    N = dev_env.n_worlds
    dev_env.reset(); host_env.reset()
    g = torch.Generator().manual_seed(4)
    modes = ["pipelined", "zero_copy", "staged"]
    for i in range(30):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g)
        dev_env.step(a.to(cuda_device))
        mode = modes[i % 3]
        # pipelined: 4 chunks of 1040 worlds, the first spanning all three maps, the others inside labyrinth's range;
        # 7 chunks put boundaries elsewhere
        h = host_env.step_host(a, mode=mode, chunks=4 if i % 2 else 7, packed=packed)
        assert torch.equal(h["obs_type"], dev_env.obs_type.cpu()), mode
        assert torch.equal(h["obs_dist"].contiguous().view(torch.int16), dev_env.obs_dist.cpu().view(torch.int16)), mode
        assert torch.equal(h["reward"], dev_env.reward.cpu()) and torch.equal(h["winner"], dev_env.winner.cpu()), mode
        assert torch.equal(h["terminated"], dev_env.terminated.cpu()) and torch.equal(h["truncated"], dev_env.truncated.cpu())
    assert torch.equal(dev_env.state, host_env.state)
    dev_env.close(); host_env.close()


def test_graph_captured_step_equals_eager_step(cuda_device):
    cmaps = [pu.named_cmap(n) for n in NAMES]
    env = CatWorlds(cmaps, (1, 37, 4096), device=cuda_device, seed=2, want_critic=True, max_step_count=40)
    N = env.n_worlds
    env.reset()
    g = torch.Generator().manual_seed(1)
    acts = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
    for _ in range(5):
        env.step(acts)
    s0 = env.state.clone()
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        env.step(acts)                      # warm-up on the capture stream
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        env.step(acts)
    for t in range(30):
        acts.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g))
        env.state.copy_(s0)
        graph.replay()
        torch.cuda.synchronize()
        replay = (env.state.clone(), env._out.clone(), env.obs_f32.clone(), env.critic_f32.clone())
        env.state.copy_(s0)
        env.step(acts)
        torch.cuda.synchronize()
        eager = (env.state, env._out, env.obs_f32, env.critic_f32)
        for r, e in zip(replay, eager):
            assert torch.equal(r, e), t
        s0 = env.state.clone()
    env.close()


def test_learner_and_per_map_evaluation(cuda_device):
    maps = [load_named_map(n) for n in NAMES]
    env = BatchedCopsThievesEnv(maps, 300, device=cuda_device, seed=1, max_step_count=30)
    assert env.num_envs == 300 and env.map_names == list(NAMES)
    assert torch.bincount(env.map_index.cpu()).tolist() == [100, 100, 100]
    assert env.render(250).shape[:2] == tuple(int(v) for v in env._cmaps[2].window)
    now = dict(random_timesteps=0, learning_starts=0, policy_freeze_duration=0, opponent_freeze_duration=0)
    learner = MAPPOLearner(env, MAPPOConfig(rollouts=16, model="mlp", kl_threshold=0.0, **now), seed=0)
    for _ in range(2):
        learner.collect()
        stats = learner.update()
    for st in stats.values():
        for v in (st.policy_loss, st.value_loss, st.entropy, st.kl):
            assert v == v and abs(v) < 1e6
    cop, thief = selfplay.evaluate_agents(env, learner, n_episodes=1)
    cop2, thief2, per_map = selfplay.evaluate_agents(env, learner, n_episodes=1, by_map=True)
    assert [e["map"] for e in per_map] == list(NAMES)
    assert sum(e["episodes"] for e in per_map) == 300                      # every world finished its one episode
    assert cop2 + thief2 == pytest.approx(1.0)
    assert cop2 == pytest.approx(sum(e["cop"] * e["episodes"] for e in per_map) / 300)
    for e in per_map:
        assert e["episodes"] == 100 and 0.0 <= e["cop"] <= 1.0 and e["cop"] + e["thief"] == pytest.approx(1.0)
    assert env.worlds.overflow_counts() == (0, 0)
    env.close()
