"""Procedural maps and the map-swap entry points without a GPU: the maze generator (deterministic per seed, spawn
regions clear of every hull, cop and thief regions connected through free space, a lossless catmap-1 round trip), the
ctypes prototypes of cat_env_create_swappable / cat_env_set_map / cat_map_blob_bytes / cat_ray_lists_device, the
blob sizing call, and clean failures (CAT_ERR_INVALID for bad arguments, CAT_ERR_CUDA without a device)."""
import ctypes as C
import json
import os
import subprocess
import sys
from collections import deque
from pathlib import Path

import numpy as np
import pytest

from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.maps import (MAZE_SPAWN_MARGIN, SHIPPED_MAPS, WALL_RADIUS, Map, compile_map, generate_maze,
                                           load_named_map)
from as_cops_and_thieves_b200.params import EnvParams
from as_cops_and_thieves_b200.worlds import _map_desc, default_blob_capacity, map_blob_bytes

ROOT = Path(__file__).resolve().parents[1]
AGENT_RADIUS = EnvParams().unit_size


def _params(**over):
    d = EnvParams().as_dict()
    d.update(over)
    return _lib.CatParams(**{n: d[n] for n, _ in _lib.CatParams._fields_})


def _arrays(cmap):
    return [np.asarray(getattr(cmap, f)) for f in ("hull_off", "vert", "normal", "edge_len", "hull_bb", "init_pos",
                                                   "region_off", "regions", "con_cell_off", "con_cell_hulls",
                                                   "view_cell_off", "view_cell_edges")]


def test_maze_is_deterministic_per_seed_and_differs_across_seeds():
    a, b = compile_map(generate_maze(7)), compile_map(generate_maze(7))
    assert a.name == "maze-7"
    for x, y in zip(_arrays(a), _arrays(b)):
        assert np.array_equal(x, y)
    verts = {compile_map(generate_maze(s)).vert.tobytes() for s in range(12)}
    assert len(verts) == 12


def test_maze_walls_are_merged_rect_blocks():
    cols, rows = 16, 9
    m = generate_maze(3, cols=cols, rows=rows)
    assert all(len(ring) == 5 for ring in m.blocks)
    cm = compile_map(m)
    assert (np.diff(cm.hull_off) == 4).all()
    # a perfect maze on cols x rows cells removes cols * rows - 1 of the interior wall segments; merging collinear runs
    # leaves fewer blocks than segments
    segments = (cols * (rows + 1) + rows * (cols + 1)) - (cols * rows - 1)
    assert cm.n_hulls < segments / 2
    # the outer boundary: the four sides of the maze's bounding box are walls along their whole length
    bb = cm.hull_bb
    x0, y0, x1, y1 = bb[:, 0].min(), bb[:, 1].min(), bb[:, 2].max(), bb[:, 3].max()
    assert ((bb[:, 0] == x0) & (bb[:, 2] - bb[:, 0] < 20) & (bb[:, 1] == y0) & (bb[:, 3] == y1)).any()
    assert ((bb[:, 1] == y0) & (bb[:, 3] - bb[:, 1] < 20) & (bb[:, 0] == x0) & (bb[:, 2] == x1)).any()


def _free(cm, x, y, clear):
    """No hull (axis-aligned rects here) within `clear` of the point."""
    bb = cm.hull_bb
    dx = np.maximum(np.maximum(bb[:, 0] - x, x - bb[:, 2]), 0.0)
    dy = np.maximum(np.maximum(bb[:, 1] - y, y - bb[:, 3]), 0.0)
    return bool((np.hypot(dx, dy) >= clear).all())


@pytest.mark.parametrize("seed", range(6))
def test_maze_spawn_regions_clear_every_hull_and_connect(seed):
    cm = compile_map(generate_maze(seed))
    clear = AGENT_RADIUS + WALL_RADIUS + MAZE_SPAWN_MARGIN
    assert cm.n_cops == 2 and cm.n_thieves == 1 and len(cm.region_off) == 4
    for x, y, w, h in cm.regions:
        assert w > 0 and h > 0
        for px in np.linspace(x, x + w, 9):
            for py in np.linspace(y, y + h, 9):
                assert _free(cm, px, py, clear - 1e-9), (seed, px, py)
    for px, py in cm.init_pos:
        assert _free(cm, px, py, clear - 1e-9)
    # free space for an agent (its disc clear of every rounded hull) on a 2-unit raster, flood-filled from the cops'
    # region: the thief's region is reached
    step = 2.0
    W, H = cm.window
    nx, ny = int(W / step), int(H / step)
    xs, ys = (np.arange(nx) + 0.5) * step, (np.arange(ny) + 0.5) * step
    bb = cm.hull_bb
    dx = np.maximum(np.maximum(bb[None, None, :, 0] - xs[:, None, None], xs[:, None, None] - bb[None, None, :, 2]), 0.0)
    dy = np.maximum(np.maximum(bb[None, None, :, 1] - ys[None, :, None], ys[None, :, None] - bb[None, None, :, 3]), 0.0)
    free = (np.hypot(dx, dy) > AGENT_RADIUS + WALL_RADIUS).all(axis=-1)

    def cell(p):
        return int(p[0] / step), int(p[1] / step)
    cop = cell(cm.regions[0][:2] + cm.regions[0][2:] / 2)
    thief = cell(cm.regions[2][:2] + cm.regions[2][2:] / 2)
    assert free[cop] and free[thief]
    seen = np.zeros_like(free)
    seen[cop] = True
    q = deque([cop])
    while q:
        i, j = q.popleft()
        for a, b in ((i + 1, j), (i - 1, j), (i, j + 1), (i, j - 1)):
            if 0 <= a < nx and 0 <= b < ny and free[a, b] and not seen[a, b]:
                seen[a, b] = True
                q.append((a, b))
    assert seen[thief]
    # far apart: the spawn cells are not neighbours
    assert np.hypot(*(cm.regions[0][:2] - cm.regions[2][:2])) > 2 * (60.0 + 16.0)


def test_maze_round_trips_through_catmap_json(tmp_path):
    m = generate_maze(11)
    path = tmp_path / "maze-11.catmap.json"
    path.write_text(json.dumps(m.to_dict()))
    for other in (Map(path), Map.from_dict(json.loads(path.read_text()), "maze-11")):
        a, b = compile_map(m), compile_map(other)
        assert a.name == b.name == "maze-11" and a.window == b.window
        for x, y in zip(_arrays(a), _arrays(b)):
            assert np.array_equal(x, y)


def test_shipped_map_round_trips_through_from_dict():
    m = load_named_map("squarinth")
    a, b = compile_map(m), compile_map(Map.from_dict(m.to_dict(), "squarinth"))
    for x, y in zip(_arrays(a), _arrays(b)):
        assert np.array_equal(x, y)


def test_default_mazes_fit_the_default_capacity():
    p = EnvParams().as_dict()
    cap = default_blob_capacity(p)
    assert cap >= max(map_blob_bytes(compile_map(load_named_map(n), name=n), p) for n in SHIPPED_MAPS)
    for seed in range(10):
        assert map_blob_bytes(compile_map(generate_maze(seed)), p) <= cap


def test_maze_argument_checks():
    with pytest.raises(ValueError, match="does not fit"):
        generate_maze(0, cols=40, rows=9)
    with pytest.raises(ValueError, match="spawn region"):
        generate_maze(0, corridor=10.0)


# ---------------------------------------------------------------------------------------------------- ABI
def test_prototypes_of_the_map_swap_entry_points():
    L = _lib.load()
    assert L.cat_env_create_swappable.argtypes == [C.POINTER(_lib.CatMapDesc), C.c_int32, C.POINTER(C.c_int32),
                                                   C.POINTER(_lib.CatParams), C.c_int32, C.c_int64, C.c_int32,
                                                   C.POINTER(C.c_void_p)]
    assert L.cat_env_set_map.argtypes == [C.c_void_p, C.c_int32, C.POINTER(_lib.CatMapDesc), C.c_void_p]
    assert L.cat_map_blob_bytes.argtypes == [C.POINTER(_lib.CatMapDesc), C.POINTER(_lib.CatParams), C.POINTER(C.c_int32)]
    assert L.cat_ray_lists_device.argtypes == L.cat_ray_lists_host.argtypes + [C.c_int32]
    header = (ROOT / "include" / "cat_b200.h").read_text()
    for decl in ("int cat_env_create_swappable(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map,\n"
                 "                             const CatParams* params, int32_t blob_capacity, int64_t gid0, int32_t device, CatEnv** out);",
                 "int cat_env_set_map(CatEnv* env, int32_t m, const CatMapDesc* desc, void* stream);",
                 "int cat_map_blob_bytes(const CatMapDesc* map, const CatParams* params, int32_t* bytes);"):
        assert decl in header


def test_map_blob_bytes():
    L = _lib.load()
    sizes = {}
    for name in SHIPPED_MAPS:
        md, keep = _map_desc(compile_map(load_named_map(name)))
        out = C.c_int32(0)
        assert L.cat_map_blob_bytes(C.byref(md), C.byref(_params()), C.byref(out)) == 0
        assert out.value > 144 and out.value % 16 == 0
        sizes[name] = out.value
    assert max(sizes, key=sizes.get) == "agh-map"
    assert default_blob_capacity(EnvParams().as_dict()) >= sizes["agh-map"]
    md, keep = _map_desc(compile_map(load_named_map("squarinth")))
    out = C.c_int32(0)
    assert L.cat_map_blob_bytes(None, C.byref(_params()), C.byref(out)) == -1
    assert L.cat_map_blob_bytes(C.byref(md), None, C.byref(out)) == -1
    assert L.cat_map_blob_bytes(C.byref(md), C.byref(_params()), None) == -1
    assert L.cat_map_blob_bytes(C.byref(md), C.byref(_params(n_rays=1000)), C.byref(out)) == -3
    # more rays: a larger direction table
    a, b = C.c_int32(0), C.c_int32(0)
    L.cat_map_blob_bytes(C.byref(md), C.byref(_params(n_rays=45)), C.byref(a))
    L.cat_map_blob_bytes(C.byref(md), C.byref(_params(n_rays=90)), C.byref(b))
    assert b.value - a.value == 45 * 16


def test_argument_validation_before_any_cuda_call():
    L = _lib.load()
    descs = [_map_desc(compile_map(load_named_map(n))) for n in ("squarinth", "agh-map")]
    maps = (_lib.CatMapDesc * 2)(*[md for md, _ in descs])
    counts = (C.c_int32 * 2)(4, 4)
    pr = _params()
    h = C.c_void_p()

    def create(m=maps, n=2, cnt=counts, p=pr, cap=1 << 16):
        return L.cat_env_create_swappable(m, n, cnt, C.byref(p) if p is not None else None, cap, 0, 0, C.byref(h))
    assert create(m=None) == -1 and b"null" in L.cat_last_error()
    assert create(cnt=None) == -1
    assert create(p=None) == -1
    assert create(n=0) == -1
    assert create(p=_params(ray_list_cell=-1.0)) == -1 and b"ray lists" in L.cat_last_error()
    assert create(cap=0) == -1
    for cap in (25000, 65535, 8):            # not a positive multiple of 16: the kernel's bulk copy of the blob needs one
        assert create(cap=cap) == -1 and b"multiple of 16" in L.cat_last_error()
    for cap in (227 * 1024 + 16, 0x7FFFFFF0):   # more than any block's shared memory: refused before any allocation
        assert create(cap=cap) == -3 and b"shared memory" in L.cat_last_error()
    assert create(cap=1024) == -3 and b"blob_capacity" in L.cat_last_error()        # smaller than agh-map's blob
    assert not h.value
    md = descs[0][0]
    assert L.cat_env_set_map(None, 0, C.byref(md), None) == -1
    grid = (C.c_double * 5)()
    n = C.c_int64(0)
    assert L.cat_ray_lists_device(None, 90, 400.0, 2.0, 0.0, C.byref(grid), None, C.byref(n), None, C.byref(n), 0) == -1
    assert L.cat_ray_lists_device(C.byref(md), 1000, 400.0, 2.0, 0.0, C.byref(grid), None, C.byref(n), None, C.byref(n), 0) == -3


_NO_DEVICE = r"""
import ctypes as C
import pytest, torch
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.maps import compile_map, generate_maze, load_named_map
from as_cops_and_thieves_b200.params import EnvParams
from as_cops_and_thieves_b200.worlds import CatWorlds, _map_desc
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
assert not torch.cuda.is_available()
L = _lib.load()
cmap = compile_map(load_named_map("squarinth"))
md, keep = _map_desc(cmap)
d = EnvParams().as_dict()
pr = _lib.CatParams(**{n: d[n] for n, _ in _lib.CatParams._fields_})
h = C.c_void_p()
cnt = (C.c_int32 * 1)(8)
assert L.cat_env_create_swappable(C.byref(md), 1, cnt, C.byref(pr), 1 << 15, 0, 0, C.byref(h)) == -2 and not h.value
grid = (C.c_double * 5)()
ns, no = C.c_int64(0), C.c_int64(0)
assert L.cat_ray_lists_device(C.byref(md), 90, 400.0, 2.0, 0.0, C.byref(grid), None, C.byref(ns), None, C.byref(no), 0) == -2
with pytest.raises(_lib.CatError, match="no CPU fallback"):
    CatWorlds(cmap, 8, swappable_maps=True)
with pytest.raises(_lib.CatError):
    BatchedCopsThievesEnv(generate_maze(1), 16, swappable_maps=True)
print("ok")
"""


def test_entry_points_fail_cleanly_without_a_device():
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


def test_python_capacity_must_be_a_multiple_of_16():
    from as_cops_and_thieves_b200.worlds import CatWorlds
    cmap = compile_map(load_named_map("squarinth"))
    for cap in (25000, 0, -16):
        with pytest.raises(ValueError, match="multiple of 16"):
            CatWorlds(cmap, 8, swappable_maps=True, map_blob_capacity=cap)
