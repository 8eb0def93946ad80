"""The renderer without a device: the argument checks of cat_renderer_create / cat_render / cat_renderer_frame_size (made
before any CUDA call), cat_ray_directions against math.cos / math.sin, the numpy ray overlay against a per-pixel Python
loop, and the loud failure of the Python renderer without a device."""
import ctypes as C
import math
import os
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np

from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.maps import compile_map, load_named_map
from as_cops_and_thieves_b200.render import RAY_COLORS, ray_directions, render_rgb
from as_cops_and_thieves_b200.worlds import _map_desc

ROOT = Path(__file__).resolve().parents[1]


def _descs(names):
    descs = [_map_desc(compile_map(load_named_map(n))) for n in names]
    arr = (_lib.CatMapDesc * len(descs))(*[md for md, _ in descs])
    return arr, [keep for _, keep in descs]


def test_renderer_create_argument_validation():
    L = _lib.load()
    maps, keep = _descs(["squarinth", "agh-map"])
    win = (C.c_int32 * 18)(*([1280, 800] * 9))
    h = C.c_void_p()

    def create(m=maps, w=win, n=2, rays=90, out=True):
        return L.cat_renderer_create(m, w, n, rays, 0, C.byref(h) if out else None)

    assert create(m=None) == -1 and b"null" in L.cat_last_error()
    assert create(w=None) == -1 and b"null" in L.cat_last_error()
    assert create(out=False) == -1 and b"null" in L.cat_last_error()
    assert create(n=0) == -1 and b"n_maps" in L.cat_last_error()
    assert create(n=-1) == -1 and b"n_maps" in L.cat_last_error()
    many = (_lib.CatMapDesc * 9)(*([maps[0]] * 9))
    assert create(m=many, n=9) == -3 and b"CAT_MAX_MAPS" in L.cat_last_error()
    for rays in (1, 0, -5, _lib.CAT_MAX_RAYS + 1):
        assert create(rays=rays) == -3 and b"n_rays" in L.cat_last_error()
    for bad in ([0, 800], [1280, 0], [8193, 800], [1280, 8193], [-1, 800]):
        assert create(w=(C.c_int32 * 4)(1280, 800, *bad)) == -1 and b"window" in L.cat_last_error()
    other = (_lib.CatMapDesc * 2)(maps[0], maps[1])
    other[1].n_cops, other[1].n_thieves = 1, 2
    assert create(m=other) == -1 and b"cops and thieves" in L.cat_last_error()
    many_agents = (_lib.CatMapDesc * 1)(maps[0])
    many_agents[0].n_cops, many_agents[0].n_thieves = 5, 4
    assert create(m=many_agents, n=1) == -3 and b"CAT_MAX_AGENTS" in L.cat_last_error()
    nohull = (_lib.CatMapDesc * 1)(maps[0])
    nohull[0].vert = None
    assert create(m=nohull, n=1) == -1 and b"hull" in L.cat_last_error()
    assert not h.value


def test_render_and_frame_size_argument_validation():
    """The checks that need only the call's own arguments; the ones that need a renderer's figures are in
    tests/test_render_gpu.py."""
    L = _lib.load()
    fake = C.create_string_buffer(256)            # never dereferenced by the checks below
    buf = C.create_string_buffer(64)
    w, h = C.c_int32(), C.c_int32()
    assert L.cat_renderer_frame_size(None, 1, C.byref(w), C.byref(h)) == -1 and b"null" in L.cat_last_error()
    assert L.cat_renderer_frame_size(fake, 1, None, C.byref(h)) == -1
    assert L.cat_renderer_frame_size(fake, 1, C.byref(w), None) == -1

    def io(**kw):
        d = dict(n_frames=1, n_elements=1, pos=C.addressof(buf), pos_stride=24, downsample=1, agent_radius=5.0,
                 frames=C.addressof(buf))
        d.update(kw)
        return _lib.CatRenderIO(**d)

    def render(r=fake, **kw):
        return L.cat_render(r, C.byref(io(**kw)), None)

    assert L.cat_render(None, C.byref(io()), None) == -1 and b"null" in L.cat_last_error()
    assert L.cat_render(fake, None, None) == -1 and b"null" in L.cat_last_error()
    cases = [
        (dict(n_frames=-1), b"n_frames"), (dict(n_elements=-1), b"n_elements"),
        (dict(downsample=0), b"downsample"), (dict(downsample=-2), b"downsample"),
        (dict(pos=None), b"null pos"), (dict(frames=None), b"null pos"),
        (dict(pos=C.addressof(buf) + 2), b"4-byte"), (dict(pos_stride=26), b"4-byte"),
        (dict(ray_dist=C.addressof(buf), ray_dist_stride=540), b"together"),
        (dict(ray_type=C.addressof(buf), ray_type_stride=270), b"together"),
        (dict(ray_dist=C.addressof(buf) + 1, ray_dist_stride=540, ray_type=C.addressof(buf), ray_type_stride=270), b"2-byte"),
        (dict(ray_dist=C.addressof(buf), ray_dist_stride=541, ray_type=C.addressof(buf), ray_type_stride=270), b"2-byte"),
        (dict(agent_radius=-1.0), b"agent_radius"), (dict(agent_radius=float("nan")), b"agent_radius"),
        (dict(agent_radius=float("inf")), b"agent_radius"),
    ]
    for kw, msg in cases:
        assert render(**kw) == -1, kw
        assert msg in L.cat_last_error(), (kw, L.cat_last_error())


def test_struct_layout_of_render_io(tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text(r"""
#include <stdio.h>
#include <stddef.h>
#include "cat_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\n", sizeof(CatRenderIO), offsetof(CatRenderIO, n_elements), offsetof(CatRenderIO, ray_type_stride),
         offsetof(CatRenderIO, agent_radius), offsetof(CatRenderIO, frames));
  return 0;
}""")
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", "-I", str(ROOT / "include"), str(probe), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    T = _lib.CatRenderIO
    assert got == [C.sizeof(T), T.n_elements.offset, T.ray_type_stride.offset, T.agent_radius.offset, T.frames.offset]


def test_ray_directions_match_math_cos_sin():
    L = _lib.load()
    out = np.zeros(2, np.float32)
    assert L.cat_ray_directions(1, _lib.np_ptr(out)) == -3 and b"n_rays" in L.cat_last_error()
    assert L.cat_ray_directions(_lib.CAT_MAX_RAYS + 1, _lib.np_ptr(out)) == -3
    assert L.cat_ray_directions(90, None) == -1
    for R in (2, 4, 8, 90, 92, 100, 128):
        u = ray_directions(R)
        step = 2.0 * math.pi / R
        want = np.array([[math.cos(i * step), math.sin(i * step)] for i in range(R)], np.float64).astype(np.float32)
        ulp = np.spacing(np.abs(want))
        assert (np.abs(u.astype(np.float64) - want) <= ulp).all(), R
        exact = [0] + ([R // 4] if R % 4 == 0 else []) + ([R // 2] if R % 2 == 0 else [])
        for i in exact:
            assert u[i, 0] == np.float32(math.cos(i * step)) and u[i, 1] == np.float32(math.sin(i * step)), (R, i)
        assert u[0, 0] == 1.0 and u[0, 1] == 0.0


# ---------------------------------------------------------------- the numpy ray overlay against a per-pixel loop
def _synthetic_map():
    """64 x 48 window, one square hull (so the walls cover part of the rays), 2 cops and 1 thief."""
    v = np.array([[40.0, 30.0], [50.0, 30.0], [50.0, 40.0], [40.0, 40.0]])
    nrm = np.array([[-1.0, 0.0], [0.0, -1.0], [1.0, 0.0], [0.0, 1.0]])   # edge i runs vert[i-1] -> vert[i]
    return SimpleNamespace(window=(64.0, 48.0), n_hulls=1, hull_off=np.array([0, 4]), vert=v, normal=nrm,
                           hull_bb=np.array([[40.0, 30.0, 50.0, 40.0]]), n_cops=2)


def _brute_rays(W, H, pos, dist, types, dirs):
    """Ray layer pixel by pixel in Python floats (fp64, no fused operations): the last (a, i) that covers a pixel."""
    img = np.zeros((W, H, 3), np.uint8)
    A, R = dist.shape
    segs = []
    for a in range(A):
        px, py = float(pos[a][0]), float(pos[a][1])
        for i in range(R):
            d = float(dist[a, i])
            segs.append((px, py, px + d * float(dirs[i, 0]), py + d * float(dirs[i, 1]), RAY_COLORS.get(int(types[a, i]))))
    for x in range(W):
        for y in range(H):
            cx, cy = x + 0.5, y + 0.5
            for px, py, qx, qy, col in reversed(segs):
                if col is None:
                    continue
                ex, ey = qx - px, qy - py
                wx, wy = cx - px, cy - py
                t = wx * ex + wy * ey
                L = ex * ex + ey * ey
                if t <= 0:
                    hit = wx * wx + wy * wy <= 0.25
                elif t >= L:
                    hit = (cx - qx) * (cx - qx) + (cy - qy) * (cy - qy) <= 0.25
                else:
                    c = wx * ey - wy * ex
                    hit = c * c <= 0.25 * L
                if hit:
                    img[x, y] = col
                    break
    return img


def _check_overlay(cmap, pos, dist, types, dirs):
    W, H = int(cmap.window[0]), int(cmap.window[1])
    with_rays = render_rgb(cmap, pos, 2.0, rays=(dist, types, dirs))
    plain = render_rgb(cmap, pos, 2.0)
    brute = _brute_rays(W, H, pos, dist, types, dirs)
    drawn = plain.any(axis=-1, keepdims=True)            # walls and agents are never black
    np.testing.assert_array_equal(with_rays, np.where(drawn, plain, brute))
    return brute


def test_ray_overlay_matches_per_pixel_loop_on_edge_cases():
    cmap = _synthetic_map()
    dirs = np.array([[1, 0], [0, 1], [-1, 0], [0, -1], [0.6, 0.8], [-0.8, 0.6]], np.float32)
    pos = np.array([[10.0, 20.0], [30.0, 10.5], [20.25, 35.0]], np.float32)
    dist = np.array([[8, 0, 3, 5, 12, 7],          # agent 0 at a pixel corner: horizontal / vertical rays have
                     [0, 6, 9, 0, 20, 4],          #   centres exactly 0.5 away on both sides; agent 1: length-0 rays
                     [30, 12, 15, 40, 25, 9]], np.float16)   # agent 2: long rays through the hull and out of the window
    types = np.array([[0, 1, 2, 4, 0, 3], [4, 0, 1, 2, 4, 0], [1, 2, 0, 4, 2, 4]], np.uint8)   # type 3: not drawn
    brute = _check_overlay(cmap, pos, dist, types, dirs)
    # the ties are drawn: centre (x + 0.5, 19.5) and (x + 0.5, 20.5) are 0.5 from agent 0's first ray
    assert (brute[12, 19] == RAY_COLORS[0]).all() and (brute[12, 20] == RAY_COLORS[0]).all()
    assert not brute[12, 21].any() and not brute[12, 18].any()
    # a length-0 ray is the disc of radius 0.5 around the agent: agent 1 at (30, 10.5) covers centres (29.5, 10.5), (30.5, 10.5)
    assert brute[29, 10].any() and brute[30, 10].any()


def test_ray_overlay_matches_per_pixel_loop_on_random_rays():
    cmap = _synthetic_map()
    rng = np.random.default_rng(7)
    R = 16
    dirs = ray_directions(R)
    pos = np.stack([rng.uniform(-5, 69, 3), rng.uniform(-5, 53, 3)], axis=1).astype(np.float32)
    dist = rng.uniform(0, 40, (3, R)).astype(np.float16)
    types = rng.choice(np.array([0, 1, 2, 4], np.uint8), (3, R))
    _check_overlay(cmap, pos, dist, types, dirs)


def test_rays_none_leaves_render_rgb_unchanged():
    cmap = compile_map(load_named_map("squarinth"))
    pos = np.array([[150.0, 150.0], [400.5, 300.25], [703.0, 702.0]], np.float32)
    a = render_rgb(cmap, pos)
    b = render_rgb(cmap, pos, 5.0, rays=None)
    np.testing.assert_array_equal(a, b)
    assert a.shape == (1280, 800, 3) and (a == 255).all(axis=-1).sum() > 0


_NO_DEVICE = r"""
import pytest, torch
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.maps import compile_map, load_named_map
from as_cops_and_thieves_b200.render import Renderer
assert not torch.cuda.is_available()
with pytest.raises(_lib.CatError, match="no CPU fallback"):
    Renderer([compile_map(load_named_map("squarinth"))], 90)
print("ok")
"""


def test_renderer_fails_loudly_without_a_device():
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
