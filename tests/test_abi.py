"""The C-ABI shared library: builds, loads, exports every symbol include/cat_b200.h declares, and
fails loudly (no CPU fallback) when there is no CUDA device.  No compute calls are made here."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from as_cops_and_thieves_b200 import _lib, build as cat_build
from as_cops_and_thieves_b200.maps import compile_map, load_named_map

ROOT = Path(__file__).resolve().parents[1]


def declared_functions():
    text = (ROOT / "include" / "cat_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?(?:int|size_t|char\s*\*|const char\s*\*)\s*\*?\s*(cat_\w+)\s*\(", text, flags=re.M)
    return sorted(set(names))


def test_library_builds_for_sm100a_and_loads():
    path = cat_build.build()
    assert path.exists()
    cmd = " ".join(cat_build.nvcc_cmd())
    assert "arch=compute_100a,code=sm_100a" in cmd and "-lineinfo" in cmd
    L = _lib.load()
    assert L.cat_abi_version() == _lib.CAT_ABI_VERSION


def test_every_declared_symbol_is_exported_and_bound():
    decl = declared_functions()
    assert len(decl) >= 15
    L = _lib.load()
    for name in decl:
        assert hasattr(L, name), f"{name} declared in include/cat_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == decl, "the ctypes binding must cover exactly the declared ABI"


def test_every_struct_field_matches_what_a_c_compiler_sees(tmp_path):
    """Compile a probe against include/cat_b200.h with gcc, generated from the binding: every ``CAT_*`` constant, and for
    every ctypes struct its size and alignment and every field's offset, size and alignment, compared with ctypes.  A
    field the header does not have under the binding's name fails to compile."""
    import subprocess
    structs = {n: T for n, T in vars(_lib).items()
               if isinstance(T, type) and issubclass(T, C.Structure) and T.__module__ == _lib.__name__}
    consts = {n: v for n, v in vars(_lib).items() if n.startswith("CAT_") and isinstance(v, int)}
    assert len(structs) >= 12 and "CAT_ABI_VERSION" in consts
    want, exprs = dict(consts), {n: n for n in consts}
    for name, T in structs.items():
        want[f"sizeof({name})"], want[f"alignof({name})"] = C.sizeof(T), C.alignment(T)
        exprs[f"sizeof({name})"], exprs[f"alignof({name})"] = f"sizeof({name})", f"_Alignof({name})"
        for f, ftype in T._fields_:
            member = f"(({name}*)0)->{f}"
            for what, expr, val in (("offsetof", f"offsetof({name}, {f})", getattr(T, f).offset),
                                    ("sizeof", f"sizeof({member})", getattr(T, f).size),
                                    ("alignof", f"__alignof__({member})", C.alignment(ftype))):
                want[f"{what}({name}.{f})"], exprs[f"{what}({name}.{f})"] = val, expr
    lines = "\n".join(f'  printf("%s %lld\\n", "{key}", (long long)({expr}));' for key, expr in exprs.items())
    probe = tmp_path / "probe.c"
    probe.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "cat_b200.h"\nint main(void) {{\n{lines}\n  return 0;\n}}\n')
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", "-I", str(ROOT / "include"), str(probe), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    got = {key: int(v) for key, v in (line.split(" ") for line in out.splitlines())}
    assert got == want
    assert _lib.CAT_ABI_VERSION == 9


def _desc(cmap):
    keep = [np.ascontiguousarray(cmap.hull_off, np.int32), np.ascontiguousarray(cmap.vert), np.ascontiguousarray(cmap.normal),
            np.ascontiguousarray(cmap.edge_len), np.ascontiguousarray(cmap.hull_bb), np.ascontiguousarray(cmap.init_pos),
            np.ascontiguousarray(cmap.region_off, np.int32), np.ascontiguousarray(cmap.regions if len(cmap.regions) else np.zeros((1, 4))),
            np.ascontiguousarray(cmap.con_cell_off, np.int32), np.ascontiguousarray(np.append(cmap.con_cell_hulls, 0), np.int32)]
    p = [_lib.np_ptr(a) for a in keep]
    md = _lib.CatMapDesc(cmap.n_hulls, cmap.n_edges, p[0], p[1], p[2], p[3], p[4], cmap.n_cops, cmap.n_thieves, p[5], p[6],
                         p[7], cmap.grid_x0, cmap.grid_y0, cmap.cell, cmap.nx, cmap.ny, p[8], p[9])
    return md, keep


def _params(**over):
    from as_cops_and_thieves_b200.params import EnvParams
    d = EnvParams().as_dict()
    d.update(over)
    return _lib.CatParams(**{n: d[n] for n, _ in _lib.CatParams._fields_})


def test_argument_validation_returns_error_codes_not_crashes():
    L = _lib.load()
    cmap = compile_map(load_named_map("squarinth"))
    md, keep = _desc(cmap)
    h = C.c_void_p()
    assert L.cat_env_create(None, None, 1, 0, 0, C.byref(h)) == -1 and b"null" in L.cat_last_error()
    pr = _params()
    assert L.cat_env_create(C.byref(md), C.byref(pr), 0, 0, 0, C.byref(h)) == -1           # n_worlds < 1
    pr = _params(n_rays=1000)
    assert L.cat_env_create(C.byref(md), C.byref(pr), 4, 0, 0, C.byref(h)) == -3           # CAT_ERR_LIMIT
    pr = _params(dt=0.0)
    assert L.cat_env_create(C.byref(md), C.byref(pr), 4, 0, 0, C.byref(h)) == -1
    assert L.cat_env_step(None, None, None, None) == -1
    assert L.cat_gae(None, None, None, None, None, None, None, 4, 4, 0.99, 0.95, None) == -1
    assert L.cat_env_destroy(None) == 0
    assert L.cat_env_state_bytes(None) == 0
    assert L.cat_env_record_layout(None, None) == -1
    assert L.cat_env_overflow_counts(None, None, 0) == -1
    assert L.cat_env_step_host(None, None, None, None, None, 0, 1, 1, None) == -1
    assert L.cat_env_packed_record_layout(None, None) == -1


def test_no_gpu_means_loud_failure_not_a_cpu_fallback():
    if torch.cuda.is_available():
        # the failure mode needs a process without a device: run this test again with every device hidden
        import os
        import subprocess
        import sys
        node = f"{Path(__file__).resolve()}::test_no_gpu_means_loud_failure_not_a_cpu_fallback"
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", node], cwd=ROOT,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
        assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout + r.stderr
        return
    L = _lib.load()
    cmap = compile_map(load_named_map("squarinth"))
    md, keep = _desc(cmap)
    pr = _params()
    h = C.c_void_p()
    rc = L.cat_env_create(C.byref(md), C.byref(pr), 8, 0, 0, C.byref(h))
    assert rc == -2 and not h.value, "cat_env_create must fail with CAT_ERR_CUDA without a device"
    assert L.cat_last_error()
    from as_cops_and_thieves_b200.worlds import CatWorlds
    with pytest.raises(_lib.CatError, match="no CPU fallback"):
        CatWorlds(cmap, 8)
    from as_cops_and_thieves_b200.env import SimpleEnv, BatchedCopsThievesEnv
    with pytest.raises(_lib.CatError):
        SimpleEnv(load_named_map("squarinth"))
    with pytest.raises(_lib.CatError):
        BatchedCopsThievesEnv(load_named_map("squarinth"), 16)
    from as_cops_and_thieves_b200.gae import compute_gae
    with pytest.raises(_lib.CatError):
        compute_gae(torch.zeros(4, 4), torch.zeros(4, 4, dtype=torch.bool), torch.zeros(4, 4), torch.zeros(4))


def test_product_package_never_imports_the_oracle():
    pkg = ROOT / "as_cops_and_thieves_b200"
    for f in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list((ROOT / "include").glob("*.h")):
        text = f.read_text()
        assert "cat_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f
