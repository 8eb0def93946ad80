"""Mixed-map environments without a device: argument checks of cat_env_create_multi (made before any CUDA call), the
loud failure of the mixed-map Python faces, and the per-map world split."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import pytest

from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.env import split_worlds
from as_cops_and_thieves_b200.maps import compile_map, load_named_map
from as_cops_and_thieves_b200.params import EnvParams
from as_cops_and_thieves_b200.worlds import _map_desc

ROOT = Path(__file__).resolve().parents[1]


def _params():
    d = EnvParams().as_dict()
    return _lib.CatParams(**{n: d[n] for n, _ in _lib.CatParams._fields_})


def _descs(names):
    descs = [_map_desc(compile_map(load_named_map(n))) for n in names]
    arr = (_lib.CatMapDesc * len(descs))(*[md for md, _ in descs])
    return arr, [keep for _, keep in descs]


def test_create_multi_argument_validation():
    L = _lib.load()
    maps, keep = _descs(["squarinth", "agh-map"])
    pr = _params()
    h = C.c_void_p()
    counts = (C.c_int32 * 9)(*([4] * 9))

    def create(m, n, cnt, p=pr):
        return L.cat_env_create_multi(m, n, cnt, C.byref(p) if p is not None else None, 0, 0, C.byref(h))

    assert create(None, 2, counts) == -1 and b"null" in L.cat_last_error()
    assert create(maps, 2, None) == -1
    assert create(maps, 2, counts, p=None) == -1
    assert L.cat_env_create_multi(maps, 2, counts, C.byref(pr), 0, 0, None) == -1
    assert create(maps, 0, counts) == -1 and b"n_maps" in L.cat_last_error()
    assert create(maps, -3, counts) == -1
    many = (_lib.CatMapDesc * 9)(*([maps[0]] * 9))
    assert create(many, 9, counts) == -3 and b"CAT_MAX_MAPS" in L.cat_last_error()   # CAT_ERR_LIMIT
    assert _lib.CAT_MAX_MAPS == 8
    for bad in ([4, 0], [0, 4], [4, -1]):
        assert create(maps, 2, (C.c_int32 * 2)(*bad)) == -1 and b"n_worlds" in L.cat_last_error()
    # different teams: 1 cop + 2 thieves next to 2 cops + 1 thief (the same agent count)
    other = (_lib.CatMapDesc * 2)(maps[0], maps[1])
    other[1].n_cops, other[1].n_thieves = 1, 2
    assert create(other, 2, (C.c_int32 * 2)(4, 4)) == -1 and b"cops and thieves" in L.cat_last_error()
    # a map the single-map call refuses is refused in any position of the list
    pr_bad = _params()
    pr_bad.n_rays = 1000
    assert create(maps, 2, (C.c_int32 * 2)(4, 4), p=pr_bad) == -3
    assert not h.value
    assert L.cat_env_map_info(None, 0, None) == -1


def test_split_worlds():
    assert split_worlds(16384, 5) == [3277, 3277, 3277, 3277, 3276]
    assert split_worlds(10, 3) == [4, 3, 3]
    assert split_worlds(7, 1) == [7]
    assert sum(split_worlds(4134, 3)) == 4134
    with pytest.raises(ValueError):
        split_worlds(2, 3)
    with pytest.raises(ValueError):
        split_worlds(8, 0)


_NO_DEVICE = r"""
import pytest, torch
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.maps import compile_map, load_named_map
from as_cops_and_thieves_b200.worlds import CatWorlds
assert not torch.cuda.is_available()
maps = [load_named_map("squarinth"), load_named_map("agh-map")]
with pytest.raises(_lib.CatError, match="no CPU fallback"):
    BatchedCopsThievesEnv(maps, 16)
with pytest.raises(_lib.CatError, match="no CPU fallback"):
    CatWorlds([compile_map(m) for m in maps], [8, 8])
print("ok")
"""


def test_mixed_map_env_fails_loudly_without_a_device():
    """Run in a child process that sees no device, so the check holds on machines with a GPU too."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
