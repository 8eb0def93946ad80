"""Final observations without a GPU: the CatStepIO fields that carry them (what a C compiler sees), the ABI version, and
the learner's refusal to bootstrap time limits from an environment that does not keep final observations."""
import ctypes as C
import subprocess
from pathlib import Path

import pytest
import torch

from as_cops_and_thieves_b200 import _lib, mappo

ROOT = Path(__file__).resolve().parents[1]
FIELDS = ("record_packed_types", "final_record", "final_record_world_stride", "final_obs_f32", "final_state_f32",
          "final_critic_f32")


def test_final_output_fields_match_what_a_c_compiler_sees(tmp_path):
    probe = tmp_path / "probe.c"
    offs = " ".join("%zu" for _ in FIELDS)
    args = ", ".join(f"offsetof(CatStepIO, {f})" for f in FIELDS)
    probe.write_text(f"""
#include <stdio.h>
#include <stddef.h>
#include "cat_b200.h"
int main(void) {{
  printf("%d %zu {offs}\\n", CAT_ABI_VERSION, sizeof(CatStepIO), {args});
  return 0;
}}""")
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", "-I", str(ROOT / "include"), str(probe), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [_lib.CAT_ABI_VERSION, C.sizeof(_lib.CatStepIO)] + [getattr(_lib.CatStepIO, f).offset for f in FIELDS]
    assert got == want
    assert _lib.CAT_ABI_VERSION == 8
    # appended after record_packed_types: every field an ABI 7 caller knows keeps its offset
    names = [n for n, _ in _lib.CatStepIO._fields_]
    assert names[-len(FIELDS):] == list(FIELDS)


def test_final_outputs_default_to_null():
    io = _lib.CatStepIO()
    assert io.final_record is None and io.final_obs_f32 is None and io.final_state_f32 is None and io.final_critic_f32 is None
    assert io.final_record_world_stride == 0


class _FakeEnv:
    """Just enough of BatchedCopsThievesEnv to construct a learner on the CPU."""
    possible_agents = ["cop_0", "cop_1", "thief_0"]
    num_envs, state_dim, device = 4, 1090, torch.device("cpu")
    final = None

    class worlds:
        R = 90

    def critic(self):
        return torch.zeros(4, 4, 90)

    def final_critic(self):
        return self.final

    def final_state(self):
        return self.final


@pytest.mark.parametrize("model", ["lstm", "mlp"])
def test_time_limit_bootstrap_needs_final_observations(model):
    assert mappo.MAPPOConfig().time_limit_bootstrap is False
    env = _FakeEnv()
    mappo.MAPPOLearner(env, mappo.MAPPOConfig(rollouts=16, model=model), seed=0)      # off: no requirement
    with pytest.raises(ValueError, match="final observations"):
        mappo.MAPPOLearner(env, mappo.MAPPOConfig(rollouts=16, model=model, time_limit_bootstrap=True), seed=0)
    env.final = torch.zeros(4, 4, 90) if model == "lstm" else torch.zeros(4, 1090)
    lrn = mappo.MAPPOLearner(env, mappo.MAPPOConfig(rollouts=16, model=model, time_limit_bootstrap=True), seed=0)
    assert lrn._final_value_input().shape == (4, lrn.n_value_in)
