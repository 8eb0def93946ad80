"""Scripted agents without a GPU: the controllers' rules on hand-built observations (scripts_reference.decide_numpy),
cat_script_random against the oracle's Philox (its counters apart from the spawn and parameter streams, its draws
uniform), the argument checks of cat_env_attach_scripts that need no environment, and the Python-side validation and
decoding of scripts.py."""
import ctypes as C
import subprocess
from fractions import Fraction
from pathlib import Path

import numpy as np
import pytest
import torch
from scipy import stats

from as_cops_and_thieves_b200 import _lib, scripts
from scripts_reference import ACT, axis_ray, decide_numpy, quadrant, random_action, script_counter

ROOT = Path(__file__).resolve().parents[1]
WALL, COP, THIEF, EMPTY = 0, 1, 2, 4


def _obs(R, fill_d=1000, fill_t=WALL):
    return np.full(R, fill_d, np.uint16), np.full(R, fill_t, np.uint8)


def _split(byte):
    return byte & 3, (byte >> 2) & 3, (byte >> 4) & 3


# ---------------------------------------------------------------------------------------------- geometry of the rules
@pytest.mark.parametrize("R", [90, 64, 37])
def test_quadrants_round_half_up(R):
    for i in range(R):
        x = Fraction(4 * i, R)
        want = int(x + Fraction(1, 2)) % 4          # floor(x + 1/2): halves go up
        assert quadrant(i, R) == want, (R, i)
    for q in range(4):
        assert quadrant(axis_ray(q, R), R) == q, "an axis ray lies in its own quadrant"


@pytest.mark.parametrize("R,first", [(90, (0, 12, 34, 57, 79)), (64, (0, 8, 24, 40, 56)), (37, (0, 5, 14, 24, 33))])
def test_quadrant_boundaries(R, first):
    """``first``: the first ray of quadrants 0 (ray 0), 1, 2, 3 and of quadrant 0 again after the wrap."""
    for k, i in enumerate(first):
        q = k % 4
        assert quadrant(i, R) == q
        if i > 0:
            assert quadrant(i - 1, R) == (q - 1) % 4


@pytest.mark.parametrize("R", [90, 64, 37])
def test_chase_moves_along_the_target_quadrant(R):
    for i in range(R):
        d, t = _obs(R)
        d[i], t[i] = 50, THIEF
        _, chase, _ = _split(decide_numpy(d, t, True, 1, 2, 3, 4, 0, R))
        assert chase == ACT[quadrant(i, R)]
        d[i], t[i] = 50, COP               # a teammate is not a cop's target: nothing seen
        rnd, chase, evade = _split(decide_numpy(d, t, True, 1, 2, 3, 4, 0, R))
        assert chase == rnd and evade == rnd


def test_distance_ties_go_to_the_lower_index():
    R = 90
    d, t = _obs(R)
    for i in (30, 70):                     # quadrant 1 (+y) and 3 (-y), same distance
        d[i], t[i] = 200, COP
    assert _split(decide_numpy(d, t, False, 0, 0, 0, 0, 2, R))[1] == ACT[1]
    d[70] = 199                            # strictly closer now
    assert _split(decide_numpy(d, t, False, 0, 0, 0, 0, 2, R))[1] == ACT[3]


def test_evade_scores_a_target_on_an_axis_ray_as_zero():
    R = 64
    d, t = _obs(R, 100)
    d[0], t[0] = 40, THIEF                 # closest target: quadrant 0, so evade prefers 2 (-x), then 1, then 3
    d[axis_ray(2, R)], t[axis_ray(2, R)] = 900, THIEF   # the far axis ray sees another target: score 0
    d[axis_ray(1, R)] = 300
    d[axis_ray(3, R)] = 400
    _, chase, evade = _split(decide_numpy(d, t, True, 0, 0, 0, 0, 1, R))
    assert chase == ACT[0] and evade == ACT[3]


def test_evade_prefers_the_opposite_quadrant_then_left_then_right_on_ties():
    R = 90
    for qs in range(4):
        d, t = _obs(R, 500, EMPTY)
        i = axis_ray(qs, R)
        d[i], t[i] = 60, COP
        _, chase, evade = _split(decide_numpy(d, t, False, 0, 0, 0, 0, 2, R))
        assert chase == ACT[qs] and evade == ACT[(qs + 2) % 4]
        d[axis_ray((qs + 2) % 4, R)] = 100          # the opposite quadrant is shorter: left and right tie, left wins
        _, _, evade = _split(decide_numpy(d, t, False, 0, 0, 0, 0, 2, R))
        assert evade == ACT[(qs + 1) % 4]
        d[axis_ray((qs + 3) % 4, R)] = 501          # strictly largest
        _, _, evade = _split(decide_numpy(d, t, False, 0, 0, 0, 0, 2, R))
        assert evade == ACT[(qs + 3) % 4]


def test_nothing_seen_falls_back_to_random():
    R = 37
    d, t = _obs(R, 800, EMPTY)
    for step in range(20):
        b = decide_numpy(d, t, False, 9, 11, 2, step, 2, R)
        rnd = random_action(9, 11, 2, step, 2)
        assert _split(b) == (rnd, rnd, rnd)


def test_teammates_are_obstacles_not_targets():
    R = 90
    d, t = _obs(R, 300)
    d[5], t[5] = 80, THIEF                  # a cop sees the thief in quadrant 0
    d[axis_ray(2, R)], t[axis_ray(2, R)] = 10, COP      # a teammate right behind: an obstacle 10 away
    d[axis_ray(1, R)] = 120
    d[axis_ray(3, R)] = 90
    _, chase, evade = _split(decide_numpy(d, t, True, 0, 0, 0, 0, 0, R))
    assert chase == ACT[0] and evade == ACT[1]
    d[5], t[5] = 80, COP                    # only teammates in view: nothing seen
    rnd, chase, evade = _split(decide_numpy(d, t, True, 0, 0, 0, 0, 0, R))
    assert chase == evade == rnd


# ---------------------------------------------------------------------------------------------- cat_script_random
def _probe(tmp_path, body: str) -> list:
    src = tmp_path / "probe.c"
    src.write_text(f'#include <stdio.h>\n#include "cat_philox.h"\nint main(void) {{\n{body}\nreturn 0;\n}}\n')
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", "-std=gnu11", "-I", str(ROOT / "include"), str(src), "-o", str(exe), "-lm"], check=True)
    return subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()


def test_script_random_matches_the_oracle_philox(tmp_path):
    cases = [(0, 0, 0, 0, 0), (7, 5, 1, 3, 2), (2 ** 40 + 3, 2 ** 33 + 17, 9, 399, 1),
             (0xFFFFFFFFFFFFFFFF, 123456, 0xFFFFFFFF, 0x7FFFFFFF, 7), (3, 4, 5, 2 ** 28 + 6, 0)]
    body = "\n".join(f'printf("%u\\n", cat_script_random({s}ull, {g}ull, {e}u, {n}u, {a}u));' for s, g, e, n, a in cases)
    got = [int(x) for x in _probe(tmp_path, body)]
    assert got == [random_action(s, g, e, n, a) for s, g, e, n, a in cases]


def test_script_counters_are_disjoint_from_spawns_and_parameter_draws():
    spawn = {(agent << 8) | t for agent in range(8) for t in range(256)}      # region pick and every try
    params = {0xFF00 | j for j in range(2)}
    steps = list(range(0, 4096)) + [2 ** 27 - 1, 2 ** 28 - 1, 2 ** 28, 2 ** 31 - 1]
    script = {script_counter(s, a) for s in steps for a in range(8)}
    assert not script & spawn and not script & params and not spawn & params
    assert all(c & 0x80000000 for c in script)
    assert max(spawn) < 0x800 and min(script) >= 0x80000000
    # one counter per (step_count mod 2^28, agent): no two agents or steps of an episode share a draw
    assert len({script_counter(s, a) for s in range(4096) for a in range(8)}) == 4096 * 8


def test_script_random_is_uniform():
    draws = np.array([random_action(12345, g, 1 + g % 5, s, a) for g in range(40) for s in range(50) for a in range(3)])
    assert set(np.unique(draws)) == {0, 1, 2, 3}
    assert stats.chisquare(np.bincount(draws, minlength=4)).pvalue > 1e-3
    # agents of one world at one step draw independently
    same = np.mean([random_action(1, g, 1, 0, 0) == random_action(1, g, 1, 0, 1) for g in range(2000)])
    assert abs(same - 0.25) < 0.04


# ---------------------------------------------------------------------------------------------- C ABI and Python checks
def test_attach_checks_the_environment_first():
    assert "cat_env_attach_scripts" in _lib.EXPORTS
    L = _lib.load()
    io = _lib.CatScriptIO(1 << 12, 1 << 13)
    assert L.cat_env_attach_scripts(None, C.byref(io)) == -1
    assert b"null env" in L.cat_last_error()
    assert L.cat_env_attach_scripts(None, None) == -1


def test_binding_constants_match_the_module():
    assert (_lib.CAT_SCRIPT_NONE, _lib.CAT_SCRIPT_RANDOM, _lib.CAT_SCRIPT_CHASE, _lib.CAT_SCRIPT_EVADE) == (0, 1, 2, 3)
    assert C.sizeof(_lib.CatScriptIO) == 16
    assert scripts.MODES == {"none": 0, "random": 1, "chase": 2, "evade": 3}
    assert all(scripts.mode_name(c) == n for n, c in scripts.MODES.items())


@pytest.mark.parametrize("bad", ["sneak", "", 4, -1, 2.0, True, None])
def test_bad_modes_are_refused(bad):
    with pytest.raises(ValueError):
        scripts.mode_code(bad)


def test_modes_masks_and_agent_names_are_checked():
    scripts.check_modes(torch.tensor([[0, 1], [2, 3]], dtype=torch.uint8))
    for bad in (torch.tensor([4], dtype=torch.uint8), torch.tensor([-1]), torch.tensor([1.0]), torch.tensor([True])):
        with pytest.raises(ValueError):
            scripts.check_modes(bad)
    assert scripts.check_mask(np.array([True, False, True]), 3).tolist() == [True, False, True]
    with pytest.raises(ValueError, match="bool"):
        scripts.check_mask(torch.tensor([1, 0, 1]), 3)
    with pytest.raises(ValueError, match="entries"):
        scripts.check_mask(torch.ones(4, dtype=torch.bool), 3)
    agents = ["cop_0", "cop_1", "thief_0"]
    assert scripts.agent_modes({"thief_0": "evade", "cop_1": 2}, agents) == {2: 3, 1: 2}
    with pytest.raises(ValueError, match="unknown agent"):
        scripts.agent_modes({"robber": "evade"}, agents)
    with pytest.raises(ValueError):
        scripts.agent_modes({"thief_0": "hide"}, agents)
    assert scripts.parse_spec("thief_0=evade, cop_0=chase") == {"thief_0": "evade", "cop_0": "chase"}
    assert scripts.parse_spec("") == {}
    for bad in ("thief_0", "=evade", "thief_0=hide"):
        with pytest.raises(ValueError):
            scripts.parse_spec(bad)


def test_decode_picks_each_agents_controller():
    rnd, chase, evade = 1, 2, 3
    dec = torch.tensor([[rnd | chase << 2 | evade << 4] * 4], dtype=torch.uint8)
    modes = torch.tensor([[0, 1, 2, 3]], dtype=torch.uint8)
    assert scripts.decode(dec, modes).tolist() == [[-1, rnd, chase, evade]]
    assert scripts.decode(dec, modes).dtype == torch.int64
