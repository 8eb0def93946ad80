"""Swapping maps of a live environment on the GPU: the device ray-list builder against the host reference word for word,
swappable environments after cat_env_set_map against freshly created ones bit for bit (eagerly, in a replayed CUDA graph
and in a MAPPO rollout graph), the error paths, device memory over many swaps, and the renderer / recorder after a
swap."""
import ctypes as C

import numpy as np
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import SHIPPED_MAPS, compile_map, generate_maze, load_named_map
from as_cops_and_thieves_b200.params import EnvParams
from as_cops_and_thieves_b200.render import TrajectoryRecorder, render_rgb
from as_cops_and_thieves_b200.worlds import CatWorlds, _map_desc, map_blob_bytes

pytestmark = pytest.mark.gpu


def _lists(fn, cmap, R, cell, device=None):
    """(grid, slots, ovf) from cat_ray_lists_host / cat_ray_lists_device with the default sensor parameters."""
    L = _lib.load()
    p = EnvParams()
    md, keep = _map_desc(cmap)
    grid = (C.c_double * 5)()
    ns, no = C.c_int64(0), C.c_int64(0)
    extra = () if device is None else (device,)
    args = (C.byref(md), R, p.ray_length, p.wall_radius + p.ray_radius, cell, C.byref(grid))
    _lib.check(fn(*args, None, C.byref(ns), None, C.byref(no), *extra), "size")
    if device is None:
        slots, ovf = np.zeros(ns.value, np.uint32), np.zeros(no.value, np.uint32)
        _lib.check(fn(*args, _lib.np_ptr(slots), C.byref(ns), _lib.np_ptr(ovf), C.byref(no)), "fill")
    else:
        s = torch.zeros(ns.value, dtype=torch.int32, device=f"cuda:{device}")
        o = torch.zeros(no.value, dtype=torch.int32, device=f"cuda:{device}")
        _lib.check(fn(*args, s.data_ptr(), C.byref(ns), o.data_ptr(), C.byref(no), *extra), "fill")
        slots, ovf = s.cpu().numpy().view(np.uint32), o.cpu().numpy().view(np.uint32)
    return list(grid), slots, ovf


def _assert_lists_equal(cmap, R, cell, dev):
    L = _lib.load()
    gh, sh, oh = _lists(L.cat_ray_lists_host, cmap, R, cell)
    gd, sd, od = _lists(L.cat_ray_lists_device, cmap, R, cell, dev)
    assert gh == gd, (cmap.name, R, cell, "grid")
    assert sh.shape == sd.shape and np.array_equal(sh, sd), (cmap.name, R, cell, "slots", int((sh != sd).sum()))
    assert oh.shape == od.shape and np.array_equal(oh, od), (cmap.name, R, cell, "overflow", oh.shape, od.shape)


@pytest.mark.parametrize("name", SHIPPED_MAPS)
@pytest.mark.parametrize("cell", [0.0, 6.8, 13.6, 48.0])
@pytest.mark.parametrize("R", [90, 45, 128])
def test_device_lists_equal_host_lists(cuda_device, name, cell, R):
    _assert_lists_equal(pu.named_cmap(name), R, cell, cuda_device.index or 0)


def test_device_lists_equal_host_lists_mazes(cuda_device):
    for seed in range(10):
        cmap = compile_map(generate_maze(seed))
        for cell in (0.0, 48.0):
            _assert_lists_equal(cmap, 90, cell, cuda_device.index or 0)
    # a larger, finer maze of many edges
    _assert_lists_equal(compile_map(generate_maze(99, cols=30, rows=16, corridor=30.0, wall=10.0)), 90, 0.0,
                        cuda_device.index or 0)


def _max_list_length(slots, ovf):
    n_max = 0
    for s in np.nonzero(slots.reshape(-1, 4)[:, 3] & 0x80000000)[0]:
        n, o = 3, int(slots[4 * s + 3] & 0x7FFFFFFF)
        while ovf[o + 3] & 0x80000000 and ovf[o + 3] != 0x7F80FFFF:
            n, o = n + 3, int(ovf[o + 3] & 0x7FFFFFFF)
        n_max = max(n_max, n + int((ovf[o:o + 4] != 0x7F80FFFF).sum()))
    return n_max


def test_long_lists_take_the_global_paths(cuda_device):
    """A dense maze (3424 edges) with coarse cells: lists longer than the on-chip sort capacity (256 entries) are sorted
    in global memory, and at 200-unit cells some cells have more candidates than are staged in shared memory (2048);
    the words still equal the host's."""
    dense = compile_map(generate_maze(5, cols=56, rows=32, corridor=18.0, wall=4.0))
    assert dense.n_edges > 3000
    for cell in (96.0, 200.0):
        _, slots, ovf = _lists(_lib.load().cat_ray_lists_host, dense, 90, cell)
        assert _max_list_length(slots, ovf) > 256
        _assert_lists_equal(dense, 90, cell, cuda_device.index or 0)
    _assert_lists_equal(pu.named_cmap("agh-map"), 90, 96.0, cuda_device.index or 0)


# ---------------------------------------------------------------------------------------------------- swap equivalence
def _same(a: CatWorlds, b: CatWorlds, what: str):
    N = a.n_worlds
    assert torch.equal(a.state.view(N, -1), b.state.view(N, -1)), f"{what}: state"
    assert torch.equal(a._out.view(N, -1), b._out.view(N, -1)), f"{what}: records"
    for name in ("obs_f32", "state_f32", "critic_f32", "final_obs_f32", "final_state_f32", "final_critic_f32"):
        x, y = getattr(a, name), getattr(b, name)
        if x is not None:
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), f"{what}: {name}"
    if a._final_out is not None:
        assert torch.equal(a._final_out, b._final_out), f"{what}: final records"


def _run_lockstep(a, b, steps, seed=7, check_counts=True):
    g = torch.Generator().manual_seed(seed)
    caps = touts = 0
    for t in range(steps):
        act = torch.randint(0, 4, (a.n_worlds, a.A), dtype=torch.uint8, generator=g).to(a.device)
        a.step(act)
        b.step(act)
        _same(a, b, f"step {t}")
        caps += int((b.terminated.bool() & ~b.truncated.bool()).sum())
        touts += int(b.truncated.sum())
    if check_counts:
        assert caps > 0 and touts > 0, (caps, touts)


KW = dict(seed=5, gid0=11, want_critic=True, max_step_count=40)


def _restart_like(sw: CatWorlds, fresh: CatWorlds):
    """Give the swapped environment the freshly created one's state, then reset both.  set_map leaves world state to
    the caller, and with pymunk's stale shape cache a reset depends on the positions before it; from the same state the
    two must then behave identically, which is what makes the swapped map indistinguishable from a fresh one."""
    sw.state.copy_(fresh.state)
    for name in ("_final_out", "final_obs_f32", "final_state_f32", "final_critic_f32"):   # written only where a world ends
        if getattr(sw, name) is not None:
            getattr(sw, name).copy_(getattr(fresh, name))
    sw.reset()
    fresh.reset()
    _same(sw, fresh, "reset")
    # random walks rarely end in a capture within a few dozen steps: in every 8th world put cop_0 10 units from the
    # thief (inside the termination radius), the same in both, so captures and timeouts both occur
    pos = fresh.get_state()["pos"]
    pos[::8, 0] = pos[::8, -1] + torch.tensor([10.0, 0.0], device=pos.device)
    for w in (sw, fresh):
        w.set_state(pos=pos)


def test_swap_equals_fresh_mixed_environment(cuda_device):
    sq, lab = pu.named_cmap("squarinth"), pu.named_cmap("labyrinth", free_spawn=True)
    maze = compile_map(generate_maze(4))
    counts = (1500, 900)
    sw = CatWorlds([sq, lab], counts, device=cuda_device, swappable_maps=True, want_final=True, **KW)
    sw.reset()
    g = torch.Generator().manual_seed(1)
    for _ in range(30):      # some history on the old map
        sw.step(torch.randint(0, 4, (sw.n_worlds, 3), dtype=torch.uint8, generator=g).to(cuda_device))
    mask = sw.set_map(1, maze)
    assert torch.equal(mask.cpu(), torch.arange(sw.n_worlds) >= counts[0])
    assert sw.cmaps[1] is maze and sw.map_info(1).n_edges == maze.n_edges
    fresh = CatWorlds([sq, maze], counts, device=cuda_device, want_final=True, **KW)
    _restart_like(sw, fresh)
    _run_lockstep(sw, fresh, 200)


def test_swap_single_map_and_back(cuda_device):
    sq, maze = pu.named_cmap("squarinth"), compile_map(generate_maze(8))
    N = 3000
    sw = CatWorlds(sq, N, device=cuda_device, swappable_maps=True, **KW)
    sw.reset()
    sw.set_map(0, maze)
    for target in (maze, sq):
        if target is sq:
            sw.set_map(0, sq)
        fresh = CatWorlds(target, N, device=cuda_device, **KW)
        _restart_like(sw, fresh)
        _run_lockstep(sw, fresh, 200)
        fresh.close()
    assert sw.info.ray_list_bytes == CatWorlds(sq, 64, device=cuda_device, **KW).info.ray_list_bytes


def test_graph_replays_the_new_map(cuda_device):
    sq, lab, maze = pu.named_cmap("squarinth"), pu.named_cmap("lbirinth"), compile_map(generate_maze(12))
    counts = (700, 600)
    sw = CatWorlds([sq, lab], counts, device=cuda_device, swappable_maps=True, **KW)
    sw.reset()
    N = sw.n_worlds
    act = torch.zeros((N, 3), dtype=torch.uint8, device=cuda_device)
    s = torch.cuda.Stream(cuda_device)
    s.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(s):
        sw.step(act)                 # warm-up outside capture
    torch.cuda.current_stream(cuda_device).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        sw.step(act)
    sw.set_map(1, maze)
    fresh = CatWorlds([sq, maze], counts, device=cuda_device, **KW)
    _restart_like(sw, fresh)
    g = torch.Generator().manual_seed(3)
    for t in range(120):
        act.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device))
        graph.replay()
        fresh.step(act)
        _same(sw, fresh, f"replay {t}")


def test_rollout_graph_across_a_swap(cuda_device):
    env = BatchedCopsThievesEnv([load_named_map("squarinth"), load_named_map("lbirinth")], 512, device=cuda_device,
                                seed=1, max_step_count=50, swappable_maps=True)
    lrn = MAPPOLearner(env, MAPPOConfig(rollouts=16), seed=0)
    lrn.collect()                    # eager warm-up
    lrn.collect()                    # captured and replayed
    (uniform, graph), = lrn._graphs.items()
    assert isinstance(graph, torch.cuda.CUDAGraph)
    mask = env.set_map(1, generate_maze(21))
    assert env.map_names[1] == "maze-21" and env.maps[1].map_path == "maze-21"
    lrn.note_reset(mask)
    lrn.collect()
    assert lrn._graphs[uniform] is graph                      # replayed, not recaptured
    m = mask.to(cuda_device)
    assert lrn.mem_reset[0][m].all()
    for a in lrn.agents:
        for role in ("policy", "value"):
            h = lrn.mem[a][role + "_h"][0]                   # the state step 0 of the rollout started from
            assert not h[:, m].any(), (a, role)
    assert torch.isfinite(lrn.mem[lrn.agents[0]]["val"]).all()


# ---------------------------------------------------------------------------------------------------- errors and memory
def test_errors_leave_the_environment_on_its_old_map(cuda_device):
    sq, lab = pu.named_cmap("squarinth"), pu.named_cmap("lbirinth")
    p = EnvParams().as_dict()
    p.update(max_step_count=KW["max_step_count"])
    cap = max(map_blob_bytes(sq, p), map_blob_bytes(lab, p))
    sw = CatWorlds(sq, 1000, device=cuda_device, swappable_maps=True, map_blob_capacity=cap, **KW)
    twin = CatWorlds(sq, 1000, device=cuda_device, **KW)
    assert twin.info.map_blob_bytes == map_blob_bytes(sq, twin.params)     # the host sizing = what creation reports
    assert sw.info.map_blob_bytes == cap and sw.map_info(0).map_blob_bytes == cap
    with pytest.raises(_lib.CatError, match=r"\(-3\).*no launch shape"):     # no room left for two warps' scratch
        CatWorlds(sq, 64, device=cuda_device, swappable_maps=True, map_blob_capacity=227 * 1024, **KW)
    big = pu.named_cmap("agh-map")
    assert map_blob_bytes(big, sw.params) > cap
    with pytest.raises(_lib.CatError, match=r"\(-3\)"):
        sw.set_map(0, big)
    with pytest.raises(_lib.CatError, match=r"\(-1\)"):
        sw.set_map(0, compile_map(generate_maze(1, n_cops=1, n_thieves=1)))
    md, keep = _map_desc(lab)
    assert _lib.load().cat_env_set_map(sw._h, 1, C.byref(md), None) == -1          # bad index
    assert _lib.load().cat_env_set_map(sw._h, -1, C.byref(md), None) == -1
    assert _lib.load().cat_env_set_map(twin._h, 0, C.byref(md), None) == -1        # not swappable
    assert sw.cmaps[0] is sq
    sw.reset()
    twin.reset()
    _run_lockstep(sw, twin, 100, check_counts=False)


def test_memory_returns_after_alternating_swaps(cuda_device):
    sq = pu.named_cmap("squarinth")
    mazes = [compile_map(generate_maze(s)) for s in (30, 31)]
    sw = CatWorlds(sq, 512, device=cuda_device, swappable_maps=True, **KW)
    sw.set_map(0, mazes[0])
    torch.cuda.synchronize()
    level = torch.cuda.mem_get_info(cuda_device)[0]
    for i in range(20):
        sw.set_map(0, mazes[(i + 1) % 2])
    torch.cuda.synchronize()
    assert sw.cmaps[0] is mazes[0]
    assert abs(torch.cuda.mem_get_info(cuda_device)[0] - level) <= 2 << 20
    ref = CatWorlds(mazes[0], 64, device=cuda_device, **KW)
    assert sw.info.ray_list_bytes == ref.info.ray_list_bytes
    assert sw.map_info(0).ray_list_cells == ref.info.ray_list_cells


# ---------------------------------------------------------------------------------------------------- rendering
def test_renderer_and_recorder_after_a_swap(cuda_device):
    sq, maze = pu.named_cmap("squarinth"), compile_map(generate_maze(40))
    sw = CatWorlds(sq, 64, device=cuda_device, swappable_maps=True, **KW)
    sw.reset()
    sw.render_frames([0])
    rec = TrajectoryRecorder(sw, [0, 1], capacity=4)
    rec.record()
    sw.set_map(0, maze)
    frame = sw.render_frames([3])[0].cpu().numpy()
    pos = sw.positions()[3].cpu().numpy()
    ref = render_rgb(maze, pos)
    W, H = ref.shape[:2]
    assert np.array_equal(frame[:W, :H], ref)
    with pytest.raises(RuntimeError, match="replaced a map"):
        rec.frames()
    with pytest.raises(RuntimeError, match="replaced a map"):
        rec.save("/dev/null")
