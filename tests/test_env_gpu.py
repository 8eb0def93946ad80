"""GPU tests of the reference-facing surfaces (PettingZoo single world, skrl-style batched),
the flattened layouts, GAE kernels, CUDA-graph capture, checkpointing and full-size properties."""
import numpy as np
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import spaces, _lib
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv, SimpleEnv, BaseEnv
from as_cops_and_thieves_b200.gae import compute_gae
from as_cops_and_thieves_b200.maps import compile_map, load_named_map, free_space_regions, Map
from as_cops_and_thieves_b200.worlds import CatWorlds
from oracle import cat_oracle as co
from oracle.cat_oracle import Oracle

pytestmark = pytest.mark.gpu


def test_simple_env_pettingzoo_surface(cuda_device):
    """What driver.py / evaluate_agents do with the env (driver.py:57-69, eval_pfsp_agents.py:25-50)."""
    env = SimpleEnv(load_named_map("squarinth"), max_step_count=25, device=cuda_device)
    assert env.possible_agents == ["cop_0", "cop_1", "thief_0"]
    assert env.metadata["render_modes"] == ["human", "rgb_array"] and env.render_mode == "rgb_array"
    assert env.time_step == pytest.approx(1 / 60)
    assert BaseEnv.__init__.__defaults__[3] == pytest.approx(1 / 15)     # base_env.py:57 default differs
    obs, infos = env.reset(seed=3)
    assert env.agents == env.possible_agents and infos == {a: {} for a in env.agents}
    for a in env.agents:
        assert set(obs[a]) == {"distance", "object_type"}
        assert obs[a]["distance"].dtype == np.float16 and obs[a]["distance"].shape == (90,)
        assert obs[a]["object_type"].dtype == np.uint8
        assert env.observation_space(a).contains(obs[a])
        assert env.action_space(a).n == 4
    st = env.state()
    assert set(st["cop_0"]) == {"own_obj_types", "own_distances", "object_type_shared", "distance_shared", "team_positions"}
    assert st["cop_0"]["team_positions"].shape == (2, 2) and st["thief_0"]["team_positions"].shape == (1, 2)
    assert st["cop_0"]["distance_shared"] is st["cop_1"]["distance_shared"]      # aliased within a team
    flat = spaces.flatten(env.state_space, st)
    assert flat.shape == (1090,)
    winner = None
    rng = np.random.default_rng(0)
    for t in range(25):
        acts = {a: int(rng.integers(0, 4)) for a in env.agents}
        obs, rew, term, trunc, infos = env.step(acts)
        assert set(rew) == set(acts) and all(isinstance(v, float) for v in rew.values())
        if any(term.values()):
            winner = infos["cop_0"]["winner"]
            break
        assert infos["cop_0"]["winner"] is None and env.agents
    assert env.agents == [] and winner in ("cop", "thief")
    if t == 24:
        assert winner == "thief" and all(trunc.values()) and rew["thief_0"] == 1.0 and rew["cop_0"] == -1.0
    assert env.step({}) == ({}, {}, {}, {}, {})                                   # base_env.py:374-376
    img = env.render()
    assert img.shape == (1280, 800, 3)
    assert env.get_base_observation_space_structure() is env.state_space
    nested = env.get_nested_agent_observation_spaces()
    assert "cop_1_team_positions" in nested["cop_0"].spaces and len(nested["thief_0"].spaces) == 15
    obs2, _ = env.reset(seed=3)
    env.close()


def test_single_world_env_equals_oracle_trajectory(cuda_device):
    """SimpleEnv (N=1, no auto-reset) against the oracle for a whole short episode."""
    m = load_named_map("lbirinth")
    env = SimpleEnv(m, max_step_count=60, device=cuda_device)
    orc = co.Oracle(env._cmap, auto_reset=0, max_step_count=60, seed=5)
    obs, _ = env.reset(seed=5)
    ost = orc.new_state(1)
    oout = orc.reset(ost)
    assert np.array_equal(obs["cop_0"]["object_type"], oout.obs_type[0, 0])
    rng = np.random.default_rng(1)
    for t in range(60):
        a = rng.integers(0, 4, 3)
        obs, rew, term, trunc, infos = env.step({k: int(a[i]) for i, k in enumerate(env.possible_agents)})
        oout = orc.step(ost, a[None])
        mism = sum(int((obs[k]["object_type"] != oout.obs_type[0, i]).sum()) for i, k in enumerate(env.possible_agents))
        assert mism <= 2                                    # ε rays only
        np.testing.assert_allclose([rew[k] for k in env.possible_agents], oout.reward[0], atol=5e-3)
        assert term["cop_0"] == bool(oout.terminated[0]) and trunc["cop_0"] == bool(oout.truncated[0])
        if term["cop_0"]:
            break
    env.close()


def test_batched_env_skrl_surface_and_layouts(cuda_device):
    m = load_named_map("squarinth")
    N = 512
    env = BatchedCopsThievesEnv(m, N, device=cuda_device, seed=11)
    assert env.num_envs == N and env.num_agents == 3 and env.agents == env.possible_agents
    obs, infos = env.reset()
    for a in env.possible_agents:
        assert obs[a].shape == (N, 180) and obs[a].dtype == torch.float32 and obs[a].is_cuda
    assert env.state().shape == (N, 1090) and env.state_dim == 1090
    g = torch.Generator(device="cpu").manual_seed(0)
    for _ in range(5):
        actions = {a: torch.randint(0, 4, (N, 1), generator=g).to(cuda_device) for a in env.possible_agents}
        obs, rew, term, trunc, infos = env.step(actions)
    for a in env.possible_agents:
        assert rew[a].shape == (N, 1) and rew[a].dtype == torch.float32
        assert term[a].shape == (N, 1) and term[a].dtype == torch.bool and trunc[a].dtype == torch.bool
        assert infos[a]["winner"].shape == (N,)
    assert env.agents == env.possible_agents                 # never empties: auto-reset (SURVEY.md C-10)
    # flattened fp32 layouts == numpy flatten of the native outputs (SURVEY.md a-9)
    w = env.worlds
    torch.cuda.synchronize()
    od, ot = w.obs_dist.cpu().numpy(), w.obs_type.cpu().numpy()
    for i, a in enumerate(env.possible_agents):
        want = np.concatenate([od[:, i].astype(np.float32), ot[:, i].astype(np.float32)], axis=1)
        assert np.array_equal(obs[a].cpu().numpy(), want)
    sd, stp = pu.shared_merge_numpy(od, ot, 2)
    assert np.array_equal(w.shared_type.cpu().numpy(), stp)
    assert np.array_equal(w.shared_dist.cpu().numpy().view(np.uint16), sd.view(np.uint16))
    want_state = pu.flat_state_numpy(od, ot, sd, stp, w.team_pos.cpu().numpy(), 2)
    assert np.array_equal(env.state().cpu().numpy(), want_state)
    env.close()


def test_action_input_forms_are_equivalent(cuda_device):
    m = load_named_map("lbirinth")
    N = 256
    envs = [BatchedCopsThievesEnv(m, N, device=cuda_device, seed=2) for _ in range(4)]
    for e in envs:
        e.reset()
    g = torch.Generator().manual_seed(1)
    for _ in range(10):
        a = torch.randint(0, 4, (N, 3), generator=g)
        envs[0].step({k: a[:, i:i + 1].contiguous().to(cuda_device) for i, k in enumerate(envs[0].possible_agents)})
        envs[1].step(a.to(torch.uint8).to(cuda_device))
        envs[2].step(a.to(torch.int32).to(cuda_device))
        envs[3].step(a.to(torch.int64).to(cuda_device))
    torch.cuda.synchronize()
    for e in envs[1:]:
        assert torch.equal(e.worlds.state, envs[0].worlds.state)
        assert torch.equal(e.worlds.reward, envs[0].worlds.reward)
    with pytest.raises(ValueError):
        envs[1].worlds.step(torch.zeros((N, 3), dtype=torch.float32, device=cuda_device))
    for e in envs:
        e.close()


@pytest.mark.parametrize("packed", [True, False])
def test_host_buffer_step_modes_are_equivalent(cuda_device, packed):
    """CatWorlds.step_host: the pipelined path (chunked launches + DMA on a second stream, cat_env_step_host), the
    zero-copy path (kernel stores into mapped pinned host memory) and the staged path (H2D copy -> launch -> D2H
    copy) must deliver exactly the same values, equal to what a device-resident step() holds — with the records in
    their packed form (types at 2 bits, the default) and with u8 types."""
    cmap = pu.named_cmap("squarinth")
    N = 777
    envs = {m: CatWorlds(cmap, N, device=cuda_device, seed=5, want_f32=False, want_shared=False)
            for m in ("pipelined", "pipelined5", "zero_copy", "staged", "device")}
    for w in envs.values():
        w.reset()
    ref = envs["device"]
    assert ref.d2h_bytes(True) == N * 640 and ref.d2h_bytes(False) == N * 832
    g = torch.Generator().manual_seed(3)
    for i in range(60):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g)
        ref.step(a.to(cuda_device))
        out = {"pipelined": envs["pipelined"].step_host(a.pin_memory(), mode="pipelined", chunks=2, packed=packed),
               "pipelined5": envs["pipelined5"].step_host(a, mode="pipelined", chunks=5, packed=packed),
               "zero_copy": envs["zero_copy"].step_host(a.pin_memory() if i % 2 else a, mode="zero_copy", packed=packed),
               "staged": envs["staged"].step_host(a.pin_memory(), mode="staged", packed=packed)}
        for k in ("obs_dist", "obs_type", "reward", "terminated", "truncated", "winner"):
            want = getattr(ref, k).cpu().contiguous().view(torch.uint8)
            for m, h in out.items():
                assert ("obs_type_packed" in h) == packed
                assert h[k].shape == getattr(ref, k).shape
                assert torch.equal(h[k].contiguous().view(torch.uint8), want), (i, k, m)
        if packed:      # the padding of the packed record is zero: the whole buffer is deterministic
            blobs = [h["blob"] for h in out.values()]
            assert all(torch.equal(b, blobs[0]) for b in blobs[1:])
    for w in envs.values():
        assert torch.equal(w.state, ref.state)
        w.close()
    with pytest.raises(ValueError):
        CatWorlds(cmap, 8, device=cuda_device).step_host(torch.zeros((8, 3), dtype=torch.uint8), mode="carrier-pigeon")


def test_packed_records_on_a_ragged_shape(cuda_device):
    """The packed record for a shape the <3, 90> instantiation does not cover (2 cops + 1 thief... with 37 rays: the
    generic kernel, a type count that is not a multiple of 16)."""
    cmap = pu.named_cmap("squarinth")
    N = 130
    kw = dict(device=cuda_device, seed=9, want_f32=False, want_shared=False, n_rays=37)
    a_env, b_env = CatWorlds(cmap, N, **kw), CatWorlds(cmap, N, **kw)
    a_env.reset(); b_env.reset()
    g = torch.Generator().manual_seed(4)
    for i in range(25):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g)
        a_env.step(a.to(cuda_device))
        h = b_env.step_host(a, mode="zero_copy" if i % 2 else "staged", packed=True)
        assert torch.equal(h["obs_type"], a_env.obs_type.cpu())
        assert torch.equal(h["obs_dist"].contiguous().view(torch.int16), a_env.obs_dist.cpu().view(torch.int16))
        assert torch.equal(h["reward"], a_env.reward.cpu()) and torch.equal(h["winner"], a_env.winner.cpu())
    a_env.close(); b_env.close()


def test_auto_reset_emits_terminal_reward_and_new_episode_observation(cuda_device):
    m = load_named_map("squarinth")
    N = 256
    w = CatWorlds(pu.named_cmap("squarinth"), N, device=cuda_device, max_step_count=5, seed=4, want_hits=True)
    w.reset()
    a = torch.ones((N, 3), dtype=torch.uint8, device=cuda_device)
    for t in range(5):
        w.step(a)
    torch.cuda.synchronize()
    assert torch.all(w.terminated == 1) and torch.all(w.truncated == 1) and torch.all(w.winner == 1)
    assert torch.all(w.reward[:, :2] == -1.0) and torch.all(w.reward[:, 2] == 1.0)
    st = w.get_state()
    assert torch.all(st["step_count"] == 0) and torch.all(st["episode"] == 2) and torch.all(st["vel"] == 0)
    # the observation returned with the terminal step is that of the re-spawned state
    obs_after = w.obs_dist.clone()
    w.observe()
    torch.cuda.synchronize()
    assert torch.equal(obs_after, w.obs_dist)
    w.step(a)
    torch.cuda.synchronize()
    assert torch.all(w.terminated == 0) and torch.all(w.winner == -1)
    w.close()


@pytest.mark.parametrize("tma", ["0", "1"], ids=["ldg", "tma"])
def test_gae_kernels_match_oracle_and_torch(cuda_device, monkeypatch, tma):
    # "tma": the TMA-fed variant (tensor maps + mbarrier ring) for the shapes it accepts (columns % 16 == 0); the
    # other shapes exercise the fallback to the register-pipelined kernel
    monkeypatch.setenv("CAT_GAE_TMA", tma)
    g = torch.Generator().manual_seed(0)
    # T spans: one partial segment, one chunk (256 = 32 segments x 8 steps), ragged multi-chunk carries
    for T, shape in ((64, (300, 3)), (16, (1000,)), (5, (7, 1)), (1, (33,)), (256, (40,)), (257, (31, 3)), (600, (65,)),
                     (600, (64,)), (33, (16, 3)), (257, (1024,)), (32, (16,)), (1, (16,)), (96, (80,))):
        r = torch.randn((T,) + shape, generator=g)
        v = torch.randn((T,) + shape, generator=g)
        d = torch.rand((T,) + shape, generator=g) < 0.08
        lv = torch.randn(shape, generator=g)
        ret, adv = compute_gae(r.to(cuda_device), d.to(cuda_device), v.to(cuda_device), lv.to(cuda_device), 0.99, 0.95)
        M = int(np.prod(shape))
        oret, oadv = co.gae(r.reshape(T, M).numpy(), d.reshape(T, M).numpy(), v.reshape(T, M).numpy(), lv.reshape(M).numpy())
        np.testing.assert_allclose(ret.cpu().numpy().reshape(T, M), oret, rtol=2e-5, atol=2e-5)
        np.testing.assert_allclose(adv.cpu().numpy().reshape(T, M), oadv, rtol=2e-4, atol=2e-5)
        # plain PyTorch fp32 restatement of skrl's compute_gae
        a = torch.zeros(shape)
        advs = torch.zeros_like(r)
        for t in reversed(range(T)):
            nv = v[t + 1] if t < T - 1 else lv
            a = r[t] - v[t] + 0.99 * (~d[t]).float() * (nv + 0.95 * a)
            advs[t] = a
        np.testing.assert_allclose(ret.cpu().numpy(), (advs + v).numpy(), rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(adv.cpu().numpy(), ((advs - advs.mean()) / (advs.std() + 1e-8)).numpy(), rtol=1e-3, atol=1e-4)
        ret2, adv2 = compute_gae(r.to(cuda_device), d.to(cuda_device), v.to(cuda_device), lv.to(cuda_device), normalize=False)
        np.testing.assert_allclose(adv2.cpu().numpy(), advs.numpy(), rtol=1e-4, atol=1e-4)


def test_gae_statistics_buffer_protocol(cuda_device):
    """include/cat_b200.h: the stats buffer is zeroed once by its owner; every call leaves its sums in slot (calls & 1),
    the other slot and the ticket zero — no memset in front of the kernel."""
    L = _lib.load()
    g = torch.Generator().manual_seed(3)
    stats = torch.zeros(6, dtype=torch.float64, device=cuda_device)
    stream = torch.cuda.current_stream(cuda_device).cuda_stream
    # (256, 49152): the bench size, 768 TMA CTAs in about 1.3 waves drawing tickets and adding their sums
    for call, (T, M) in enumerate(((40, 4096), (7, 33), (300, 64), (64, 1600), (256, 49152)), start=1):
        r = torch.randn((T, M), generator=g).to(cuda_device)
        v = torch.randn((T, M), generator=g).to(cuda_device)
        d = (torch.rand((T, M), generator=g) < 0.05).to(torch.uint8).to(cuda_device)
        lv = torch.randn((M,), generator=g).to(cuda_device)
        ret, adv = torch.empty_like(r), torch.empty_like(r)
        _lib.check(L.cat_gae(r.data_ptr(), d.data_ptr(), v.data_ptr(), lv.data_ptr(), ret.data_ptr(), adv.data_ptr(),
                             stats.data_ptr(), T, M, 0.99, 0.95, stream), "cat_gae")
        torch.cuda.synchronize()
        words = stats.view(torch.int64).cpu()
        assert int(words[4]) == call and int(words[5]) == 0
        s = stats.cpu().numpy()
        slot = call & 1
        a64 = adv.double()
        np.testing.assert_allclose(s[2 * slot], float(a64.sum()), rtol=1e-6, atol=1e-3)   # fp32 partials per thread
        np.testing.assert_allclose(s[2 * slot + 1], float((a64 * a64).sum()), rtol=1e-6)
        assert s[2 * (1 - slot)] == 0.0 and s[2 * (1 - slot) + 1] == 0.0
        _lib.check(L.cat_adv_normalize(adv.data_ptr(), adv.numel(), stats.data_ptr(), adv.numel(), stream), "norm")
        want = (a64 - a64.mean()) / (a64.std() + 1e-8)
        np.testing.assert_allclose(adv.cpu().numpy(), want.float().cpu().numpy(), rtol=1e-4, atol=1e-5)


def test_gae_distributed_statistics_path(cuda_device):
    """compute_gae(distributed=True): the sums of the latest call are picked out of the two-slot statistics buffer on the
    device, all-reduced with the count and handed to cat_adv_normalize — a one-rank group must reproduce the local result
    on every call (odd and even: both slots)."""
    import os
    import torch.distributed as dist
    if dist.is_initialized():
        pytest.skip("a process group already exists in this process")
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=cuda_device)
    try:
        g = torch.Generator().manual_seed(5)
        for T, M in ((32, 4096), (9, 160), (64, 48)):
            r = torch.randn((T, M), generator=g).to(cuda_device)
            v = torch.randn((T, M), generator=g).to(cuda_device)
            d = (torch.rand((T, M), generator=g) < 0.05).to(cuda_device)
            lv = torch.randn((M,), generator=g).to(cuda_device)
            ret0, adv0 = compute_gae(r, d, v, lv)
            ret1, adv1 = compute_gae(r, d, v, lv, distributed=True)
            torch.testing.assert_close(ret1, ret0, rtol=0, atol=0)
            torch.testing.assert_close(adv1, adv0, rtol=1e-5, atol=1e-6)
            a = adv1.double()
            assert abs(float(a.mean())) < 1e-4 and abs(float(a.std()) - 1.0) < 1e-3
    finally:
        dist.destroy_process_group()


def test_step_is_cuda_graph_capturable(cuda_device):
    cmap = pu.named_cmap("squarinth")
    N = 1024
    a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, device=cuda_device)
    eager = CatWorlds(cmap, N, device=cuda_device, seed=8)
    graphed = CatWorlds(cmap, N, device=cuda_device, seed=8)
    eager.reset()
    graphed.reset()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        graphed.step(a)                      # warm-up on the side stream
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            graphed.step(a)
    torch.cuda.synchronize()
    eager.step(a)                            # matches the warm-up; capture itself executes nothing
    for _ in range(10):
        eager.step(a)
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager.state, graphed.state) and torch.equal(eager.obs_dist, graphed.obs_dist)
    eager.close()
    graphed.close()


def test_checkpoint_roundtrip(cuda_device):
    cmap = pu.named_cmap("lbirinth")
    a = torch.randint(0, 4, (128, 3), dtype=torch.uint8, device=cuda_device)
    w1 = CatWorlds(cmap, 128, device=cuda_device, seed=13)
    w1.reset()
    for _ in range(7):
        w1.step(a)
    sd = w1.state_dict()
    w2 = CatWorlds(cmap, 128, device=cuda_device, seed=0)
    w2.load_state_dict(sd)
    for _ in range(30):
        w1.step(a)
        w2.step(a)
    torch.cuda.synchronize()
    assert torch.equal(w1.state, w2.state) and torch.equal(w1.reward, w2.reward)
    w1.close()
    w2.close()


FULL = [("squarinth", False, 4096, 400), ("agh-map", True, 16384, 400), ("grandbyrinth", False, 16384, 400),
        ("labyrinth", True, 8192, 400)]


@pytest.mark.parametrize("name,free,N,T", FULL, ids=[c[0] for c in FULL])
def test_full_size_properties(cuda_device, name, free, N, T):
    """BASELINE.json sizes, size-independent properties (the oracle is too slow here)."""
    cmap = pu.named_cmap(name, free_spawn=free)
    w = CatWorlds(cmap, N, device=cuda_device, seed=1, want_f32=False)
    w2 = CatWorlds(cmap, N, device=cuda_device, seed=1, want_f32=False)
    w.reset()
    w2.reset()
    g = torch.Generator(device=cuda_device).manual_seed(0)
    done_total = 0
    cops_won = 0
    for t in range(T + 5):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, device=cuda_device, generator=g)
        w.step(a)
        w2.step(a)
        if t % 50 == 49 or t >= T - 1:
            d, ty = w.obs_dist.float(), w.obs_type
            # the f16 chain rounds hit point and origin separately (spacing 1.0 above 1024), so 400 can read as ~401.5
            assert torch.isfinite(d).all() and (d >= 0).all() and (d <= 403.0).all()
            assert bool(((ty == 0) | (ty == 1) | (ty == 2) | (ty == 4)).all())
            assert bool((d[ty == 4] == 400.0).all())                     # EMPTY <=> full range
            st = w.get_state()
            assert torch.isfinite(st["pos"]).all() and torch.isfinite(st["vel"]).all()
            # the 125 clamp acts on the action impulse only (entity.py:133-134); an inelastic hit from another
            # agent can add a perpendicular component afterwards, so the bound is loose
            assert float(st["vel"].norm(dim=-1).max()) <= 2 * 125.0
            assert int(st["step_count"].max()) <= 400 and int(st["step_count"].min()) >= 0
            assert bool((w.truncated <= w.terminated).all())             # timeout implies terminated (entity.py:146)
            win = w.winner
            assert bool(((win == -1) == (w.terminated == 0)).all())
            assert bool((win[w.truncated == 1] == 1).all())              # timeout -> thief wins
            # a cop never "sees" a cop as THIEF etc.: type 2 only towards the thief
            assert bool((ty[:, 2] != 2).all())                           # the only thief cannot see a thief
        done_total += int(w.terminated.sum())
        cops_won += int((w.winner == 0).sum())
    torch.cuda.synchronize()
    assert done_total >= N                                               # every world finished at least once
    assert torch.equal(w.state, w2.state) and torch.equal(w.obs_dist, w2.obs_dist)   # bitwise deterministic
    if name == "squarinth":
        p = w.get_state()["pos"]
        assert float(p.min()) > 100.0 and float(p.max()) < 705.0         # nobody tunnels out of the box
    print(name, "episodes", done_total, "captures", cops_won)
    w.close()
    w2.close()


def test_two_environments_on_different_maps_stay_usable(cuda_device):
    """ADVICE r1: the kernel's dynamic shared-memory cap is a per-function attribute; creating an environment for a
    SMALLER map must not lower it under one that is still alive (agh-map needs ~20 KB more per CTA than squarinth)."""
    big = CatWorlds(pu.named_cmap("agh-map", free_spawn=True), 256, device=cuda_device, seed=1)
    big.reset()
    small = CatWorlds(pu.named_cmap("squarinth"), 256, device=cuda_device, seed=1)
    small.reset()
    a = torch.ones((256, 3), dtype=torch.uint8, device=cuda_device)
    for _ in range(3):
        big.step(a)
        small.step(a)
    torch.cuda.synchronize()
    # (a world that ended meanwhile restarted its count: look at the maximum)
    assert int(big.get_state()["step_count"].max()) == 3 and int(small.get_state()["step_count"].max()) == 3
    big.close()
    small.step(a)           # destroying one environment leaves the other alone
    torch.cuda.synchronize()
    small.close()


def test_reset_with_a_seed_reproduces_the_spawn(cuda_device):
    """base_env.py:307-311 re-creates np_random from the seed: reset(seed=s) restarts the spawn stream.  (The reference
    itself is NOT reproducible — it draws the point from the unseeded global `random`, SURVEY.md C-7; here the Philox
    stream is keyed by (seed, world, episode), and reset(seed) restarts the episode counter.)  With the shape cache kept
    fresh the spawn depends on nothing else, so two resets agree exactly; with pymunk's stale cache (default) the
    rejection test also looks at where the OTHER agents were before the reset, so a few worlds may differ."""
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 128, device=cuda_device, seed=0, stale_shape_cache=False)
    o1, _ = env.reset(seed=42)
    first = {k: v.clone() for k, v in o1.items()}
    p1 = env.worlds.get_state()["pos"].clone()
    for _ in range(5):
        env.step(torch.ones((128, 3), dtype=torch.uint8, device=cuda_device))
    o2, _ = env.reset(seed=42)
    assert torch.equal(env.worlds.get_state()["pos"], p1)
    assert all(torch.equal(first[k], o2[k]) for k in first)
    env.reset(seed=43)
    assert not torch.equal(env.worlds.get_state()["pos"], p1)
    env.close()
    stale = BatchedCopsThievesEnv(load_named_map("squarinth"), 512, device=cuda_device, seed=0)
    stale.reset(seed=42)
    p1 = stale.worlds.get_state()["pos"].clone()
    for _ in range(5):
        stale.step(torch.ones((512, 3), dtype=torch.uint8, device=cuda_device))
    stale.reset(seed=42)
    same = (stale.worlds.get_state()["pos"] == p1).all(dim=2).all(dim=1)
    assert float(same.float().mean()) > 0.9
    stale.close()
    single = SimpleEnv(load_named_map("squarinth"), device=cuda_device, stale_shape_cache=False)
    a, _ = single.reset(seed=7)
    single.step({k: 1 for k in single.possible_agents})
    b, _ = single.reset(seed=7)
    assert all(np.array_equal(a[k]["distance"], b[k]["distance"]) for k in a)
    single.close()


def test_fresh_shape_cache_spawns_one_agent_after_the_other(cuda_device):
    """ADVICE r1: with stale_shape_cache = 0 agent j's spawn test must see the NEW positions of agents i < j (the
    reference resets them in order); the oracle does, and the kernel must land on the same points bit for bit — and
    never on top of each other."""
    import json
    m = json.loads(json.dumps(pu.random_map_json(3, n_blocks=4)))
    for a in m["agents"]:                       # one small shared region: collisions between spawns are the norm
        a["spawn_region"] = {"x": 60.0, "y": 60.0, "w": 40.0, "h": 40.0}
    import tempfile
    from as_cops_and_thieves_b200.maps import Map
    with tempfile.NamedTemporaryFile("w", suffix=".json", delete=False) as f:
        json.dump(m, f)
    cmap = compile_map(Map(f.name), name="crowded")
    N = 512
    cw = CatWorlds(cmap, N, device=cuda_device, seed=12, stale_shape_cache=0)
    orc = Oracle(cmap, seed=12, stale_shape_cache=0)
    ost = orc.new_state(N)
    for _ in range(3):
        cw.reset()
        orc.reset(ost)
        pos = cw.get_state()["pos"].cpu().numpy().astype(np.float64)
        assert np.array_equal(pos, ost.pos)
    d01 = np.linalg.norm(pos[:, 0] - pos[:, 1], axis=-1)
    d02 = np.linalg.norm(pos[:, 0] - pos[:, 2], axis=-1)
    d12 = np.linalg.norm(pos[:, 1] - pos[:, 2], axis=-1)
    # an accepted sample keeps >= 10 between centres; only the 20-tries-failed fallback (region centre) may overlap
    centre = np.array([80.0, 80.0])
    fell_back = (np.abs(pos - centre).max(axis=-1) < 1e-6).any(axis=1)
    assert (np.minimum(np.minimum(d01, d02), d12)[~fell_back] >= 10.0 - 1e-4).all()
    cw.close()
