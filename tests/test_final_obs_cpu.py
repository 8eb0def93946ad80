"""Final observations without a GPU: the CatStepIO fields that carry them (their layout is checked with every struct's in
test_abi.py), and the learner's refusal to bootstrap time limits from an environment that does not keep final
observations."""
import pytest
import torch

from as_cops_and_thieves_b200 import _lib, mappo

FIELDS = ("record_packed_types", "final_record", "final_record_world_stride", "final_obs_f32", "final_state_f32",
          "final_critic_f32")


def test_final_output_fields_come_last():
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
