"""The device renderer against render.render_rgb, bit for bit: the five maps with random, tied, negative, out-of-window
and overlapping positions; the sensor-ray overlay of live worlds; downsampling; mixed maps; out-of-range ids; graph
capture; 64-bit frame offsets; the recorder; the environments' render(); and no side effect on the environment."""
import ctypes as C

import numpy as np
import pytest
import torch

from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv, SimpleEnv
from as_cops_and_thieves_b200.maps import compile_map, load_named_map
from as_cops_and_thieves_b200.render import TrajectoryRecorder, ray_directions, redraw, render_rgb
from as_cops_and_thieves_b200.worlds import CatWorlds

pytestmark = pytest.mark.gpu

MAPS = ["squarinth", "agh-map", "labyrinth", "lbirinth", "grandbyrinth"]
_CMAPS = {}


def cmap_of(name):
    if name not in _CMAPS:
        _CMAPS[name] = compile_map(load_named_map(name))
    return _CMAPS[name]


def _positions(cmap, rng):
    """(N, 3, 2) float32: random, disc edges through pixel centres (ties), negative / out-of-window, overlapping."""
    W, H = cmap.window
    sets = [np.stack([rng.uniform(0, W, 3), rng.uniform(0, H, 3)], 1) for _ in range(6)]
    i, j = int(rng.integers(20, 1000)), int(rng.integers(20, 600))
    sets += [np.array([[i + 0.5 + 5, j + 0.5], [i + 40.5, j + 0.5 - 5], [i + 80.5 + 3, j + 0.5 + 4]]),
             np.array([[i + 0.5 - 5, j + 20.5], [i + 30.5, j + 20.5 + 5], [i + 60.5 - 4, j + 20.5 - 3]]),
             np.array([[-3.25, 100.0], [W + 3.7, 400.0], [-10.0, -10.0]]),
             np.array([[5000.0, 5000.0], [W - 0.1, H - 0.1], [2.0, H + 4.5]]),
             np.array([[300.0, 300.0], [303.0, 301.5], [301.0, 304.0]]),
             np.array([[0.0, 0.0], [W, H], [W - 6.0, -5.5]])]
    return np.stack(sets).astype(np.float32)


@pytest.mark.parametrize("name", MAPS)
def test_frames_equal_render_rgb(cuda_device, name):
    cmap = cmap_of(name)
    pos = _positions(cmap, np.random.default_rng(MAPS.index(name)))
    cw = CatWorlds(cmap, len(pos), device=cuda_device, want_f32=False, want_shared=False)
    cw.set_state(pos=torch.from_numpy(pos))
    frames = cw.render_frames().cpu().numpy()
    assert frames.shape == (len(pos), int(cmap.window[0]), int(cmap.window[1]), 3)
    for w in range(len(pos)):
        np.testing.assert_array_equal(frames[w], render_rgb(cmap, pos[w]), err_msg=f"{name} world {w}")
    cw.close()


def _live_env(name, n, steps, seed=0, device="cuda:0"):
    env = BatchedCopsThievesEnv(load_named_map(name), n, device=device, seed=seed)
    env.reset()
    g = torch.Generator(device=device).manual_seed(seed)
    for _ in range(steps):
        env.step(torch.randint(0, 4, (n, 3), device=device, generator=g, dtype=torch.uint8))
    return env


@pytest.mark.parametrize("name", ["squarinth", "agh-map"])
def test_ray_frames_equal_numpy_overlay(cuda_device, name):
    env = _live_env(name, 64, 40)
    cw = env.worlds
    worlds = [0, 7, 31, 63]
    frames = env.render_frames(worlds, rays=True).cpu().numpy()
    dist, types = (t.cpu().numpy() for t in cw.sensor_rays())
    pos = cw.get_state()["pos"].cpu().numpy()
    dirs = ray_directions(cw.R)
    for k, w in enumerate(worlds):
        ref = render_rgb(cmap_of(name), pos[w], rays=(dist[w], types[w], dirs))
        np.testing.assert_array_equal(frames[k], ref, err_msg=f"{name} world {w}")
        assert (frames[k] == (40, 40, 40)).all(-1).sum() > 0      # the overlay is there
    env.close()


def test_private_observation_is_the_next_steps_observation(cuda_device):
    env = _live_env("agh-map", 512, 30, seed=3)
    cw = env.worlds
    env.render_frames([0], rays=True)
    dist, types = (t.clone() for t in cw.sensor_rays())
    env.step(torch.randint(0, 4, (512, 3), device=cuda_device, dtype=torch.uint8))
    live = ~cw.terminated.bool()
    assert live.sum() > 400
    assert torch.equal(dist.view(torch.int16)[live], cw.obs_dist.view(torch.int16)[live])
    assert torch.equal(types[live], cw.obs_type[live])
    env.close()


def test_rendering_has_no_side_effects(cuda_device):
    a, b = _live_env("squarinth", 256, 10, seed=5), _live_env("squarinth", 256, 10, seed=5)
    wa = a.worlds
    before = [wa.state.clone(), wa._out.clone(), wa.obs_f32.clone()]
    a.render_frames(rays=True)
    a.render_frames(list(range(0, 256, 3)), rays=True, downsample=2)
    torch.cuda.synchronize()
    for x, y in zip(before, [wa.state, wa._out, wa.obs_f32]):
        assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))
    g = torch.Generator(device=cuda_device).manual_seed(11)
    for _ in range(50):
        acts = torch.randint(0, 4, (256, 3), device=cuda_device, generator=g, dtype=torch.uint8)
        a.step(acts)
        b.step(acts)
        a.render_frames([1, 2, 200], rays=True)
    torch.cuda.synchronize()
    assert torch.equal(wa.state, b.worlds.state) and torch.equal(wa._out, b.worlds._out)
    assert torch.equal(wa.obs_f32, b.worlds.obs_f32) and torch.equal(wa.critic_f32, b.worlds.critic_f32)
    a.close(); b.close()


@pytest.mark.parametrize("d", [2, 3, 4])
def test_downsample_is_a_slice_of_the_full_frame(cuda_device, d):
    env = _live_env("agh-map", 32, 20)
    full = env.render_frames(rays=True)
    small = env.render_frames(rays=True, downsample=d)
    h = d // 2
    assert small.shape[1:3] == full[:, h::d, h::d].shape[1:3]
    assert torch.equal(small, full[:, h::d, h::d])
    env.close()


def test_three_map_environment(cuda_device):
    names = ["squarinth", "agh-map", "labyrinth"]
    env = BatchedCopsThievesEnv([load_named_map(n) for n in names], [5, 6, 7], device=cuda_device, seed=2)
    env.reset()
    for _ in range(25):
        env.step(torch.randint(0, 4, (18, 3), device=cuda_device, dtype=torch.uint8))
    cw = env.worlds
    frames = env.render_frames(rays=True).cpu().numpy()
    dist, types = (t.cpu().numpy() for t in cw.sensor_rays())
    pos = cw.get_state()["pos"].cpu().numpy()
    dirs = ray_directions(cw.R)
    assert frames.shape[1:3] == (1280, 800)
    for w in range(18):
        cmap = cw.cmaps[int(cw.map_index[w])]
        W, H = int(cmap.window[0]), int(cmap.window[1])
        np.testing.assert_array_equal(frames[w, :W, :H], render_rgb(cmap, pos[w], rays=(dist[w], types[w], dirs)))
        assert not frames[w, W:].any() and not frames[w, :, H:].any()
        np.testing.assert_array_equal(env.render(w), render_rgb(cmap, pos[w]))
    env.close()


def test_out_of_range_ids_give_zero_frames(cuda_device):
    env = _live_env("squarinth", 16, 5)
    ids = torch.tensor([-1, 3, 16, 2 ** 40, 15], dtype=torch.int64, device=cuda_device)
    frames = env.render_frames(ids, rays=True)
    assert not frames[0].any() and not frames[2].any() and not frames[3].any()
    ref = env.render_frames(torch.tensor([3, 15], device=cuda_device), rays=True)
    assert torch.equal(frames[1], ref[0]) and torch.equal(frames[4], ref[1])
    # an element whose map is not one of the renderer's also gives a zero frame
    ren = env.worlds.renderer()
    bad_map = torch.full((16,), 5, dtype=torch.int64, device=cuda_device)
    assert not ren.render(env.worlds.positions(), map_of=bad_map).any()
    env.close()


def test_render_checks_that_need_the_renderer(cuda_device):
    cw = CatWorlds(cmap_of("squarinth"), 4, device=cuda_device)
    r = cw.renderer()
    L, pos, out = cw.L, cw.positions(), torch.zeros(1 << 16, dtype=torch.uint8, device=cuda_device)
    dist, types = cw.sensor_rays()

    def render(**kw):
        d = dict(n_frames=1, n_elements=4, pos=pos.data_ptr(), pos_stride=cw.info.record_words * 4, downsample=1,
                 agent_radius=5.0, frames=out.data_ptr())
        d.update(kw)
        return L.cat_render(r._h, C.byref(_lib.CatRenderIO(**d)), None)

    assert render(pos_stride=20) == -1 and b"8 * n_agents" in L.cat_last_error()
    ok_rays = dict(ray_dist=dist.data_ptr(), ray_dist_stride=cw.record_bytes, ray_type=types.data_ptr(), ray_type_stride=cw.record_bytes)
    assert render(**dict(ok_rays, ray_dist_stride=538)) == -1 and b"block" in L.cat_last_error()
    assert render(**dict(ok_rays, ray_type_stride=269)) == -1 and b"block" in L.cat_last_error()
    assert render(downsample=5000) == -1 and b"empty frame" in L.cat_last_error()
    assert render(n_frames=2 ** 31 - 1, downsample=100) == -3 and b"too many frames" in L.cat_last_error()
    assert r.frame_size(1) == (1280, 800) and r.frame_size(3) == (427, 267) and r.frame_size(4) == (320, 200)
    with pytest.raises(_lib.CatError):
        r.frame_size(2000)
    with pytest.raises(ValueError):
        r.render(pos.contiguous()[:, :, :1])
    cw.close()


def test_graph_capture_replays_to_the_eager_frames(cuda_device):
    a, b = _live_env("agh-map", 128, 5, seed=9), _live_env("agh-map", 128, 5, seed=9)
    ids = torch.tensor([0, 17, 90, 127], dtype=torch.int64, device=cuda_device)
    acts = torch.zeros((128, 3), dtype=torch.uint8, device=cuda_device)
    out = torch.zeros((4, 1280, 768, 3), dtype=torch.uint8, device=cuda_device)
    a.render_frames(ids, rays=True, out=out)          # first call outside capture: renderer and private buffer
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        a.step(acts)
        a.render_frames(ids, rays=True, out=out)
    torch.cuda.current_stream().wait_stream(s)
    b.step(acts)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        a.step(acts)
        a.render_frames(ids, rays=True, out=out)
    gen = torch.Generator(device=cuda_device).manual_seed(1)
    for _ in range(6):
        acts.copy_(torch.randint(0, 4, (128, 3), device=cuda_device, generator=gen, dtype=torch.uint8))
        g.replay()
        b.step(acts)
        assert torch.equal(out, b.render_frames(ids, rays=True))
    assert torch.equal(a.worlds.state, b.worlds.state)
    a.close(); b.close()


def test_frame_buffer_past_2_31_bytes(cuda_device):
    free, _ = torch.cuda.mem_get_info()
    if free < 8 * 2 ** 30:
        pytest.skip(f"needs 8 GB of free device memory for a 2.2 GB frame buffer, {free / 2 ** 30:.1f} GB free")
    env = _live_env("agh-map", 64, 10)
    K = 760                                           # 760 x 1280 x 768 x 3 = 2.24e9 bytes
    ids = torch.arange(K, device=cuda_device, dtype=torch.int64) % 64
    big = env.render_frames(ids, rays=True)
    assert big.numel() > 2 ** 31
    for k0 in range(0, K, 100):
        part = env.render_frames(ids[k0:k0 + 100], rays=True)
        assert torch.equal(big[k0:k0 + 100], part), k0
    env.close()


def test_recorder_frames_and_outputs(cuda_device, tmp_path):
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 64, device=cuda_device, seed=4, max_step_count=25)
    env.reset()
    worlds = [0, 5, 63]
    T = 40
    rec = TrajectoryRecorder(env, worlds, T, rays=True)
    live, outs = [], []
    cw = env.worlds
    idx = torch.tensor(worlds, device=cuda_device)
    gen = torch.Generator(device=cuda_device).manual_seed(2)
    for _ in range(T):
        env.step(torch.randint(0, 4, (64, 3), device=cuda_device, generator=gen, dtype=torch.uint8))
        rec.record()
        live.append(env.render_frames(worlds, rays=True).clone())
        outs.append([t[idx].clone() for t in (cw.reward, cw.terminated, cw.truncated, cw.winner)])
    frames = rec.frames()
    assert frames.shape[:2] == (T, 3)
    for t in range(T):
        assert torch.equal(frames[t], live[t]), t
    for field, i in (("reward", 0), ("terminated", 1), ("truncated", 2), ("winner", 3)):
        assert torch.equal(getattr(rec, field), torch.stack([o[i] for o in outs])), field
    assert rec.truncated.any()                       # episodes of 25 steps ended inside the recording
    assert torch.equal(rec.frames(10, 20, downsample=2), torch.stack(live[10:20])[:, :, 1::2, 1::2])
    path = tmp_path / "rec.npz"
    rec.save(path)
    saved = np.load(path)
    for t, k in ((0, 0), (T - 1, 2)):
        np.testing.assert_array_equal(redraw(saved, t, k), frames[t, k].cpu().numpy())
    with pytest.raises(IndexError):
        rec.record()
    env.close()


def test_env_render_equals_render_rgb(cuda_device):
    env = _live_env("labyrinth", 8, 12)
    pos = env.worlds.get_state()["pos"].cpu().numpy()
    for w in (0, 5):
        np.testing.assert_array_equal(env.render(w), render_rgb(cmap_of("labyrinth"), pos[w]))
    env.close()
    se = SimpleEnv(load_named_map("agh-map"), device=cuda_device)
    se.reset(seed=1)
    for _ in range(15):
        se.step({a: 2 for a in se.agents})
    img = se.render()
    np.testing.assert_array_equal(img, render_rgb(cmap_of("agh-map"), se._w.get_state()["pos"][0].cpu().numpy()))
    se.close()
