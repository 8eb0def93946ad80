"""PFSP self-play bookkeeping and the batched evaluator (SURVEY.md §8 f-2).

Host-side mirror of the reference's archive / opponent-sampling / evaluation helpers, same function names,
argument meaning and on-disk format, so the reference's ``self_play_driver.py`` logic ports line by line:

* ``load_win_rates`` / ``save_win_rates`` / ``update_policy_win_rate`` / ``add_policy_to_archive`` /
  ``get_latest_policy_from_archive`` / ``sample_policy_from_archive``
  — ``/root/reference/src/utils/policy_archive_utils.py:11-199`` (``win_rates.json`` with a bounded window of
  recent outcomes per archived policy; PFSP weight ``max(1e-3, 1 - 2*|win_rate - 0.5|)``, ``:173-176``);
* ``evaluate_agents`` — ``/root/reference/src/utils/eval_pfsp_agents.py:7-59``, but batched: instead of
  ``n_episodes`` serial episodes of one world it plays every world of the batched environment until each has
  finished ``episodes_per_world`` episodes and counts ``infos["winner"]`` on the device, which turns the
  reference's 5-episode estimate into one over thousands of episodes for the same wall-clock;
* ``evaluate_agent`` / ``self_play_iteration`` — the control flow of
  ``/root/reference/src/utils/agent_learning_utils.py:233-380`` and
  ``/root/reference/src/training/orchestration.py:100-249`` over ``MAPPOLearner``.

Nothing here is on the GPU hot path; it decides WHICH weights the hot path runs.
"""
from __future__ import annotations

import json
import random
import shutil
from collections import deque
from pathlib import Path
from types import SimpleNamespace
from typing import Dict, Optional, Tuple

WIN_RATES_FILENAME = "win_rates.json"
DEFAULT_WIN_RATE = 0.5

#: ``/root/reference/src/configs/training_config.py:3-12``
TrainingConfig = SimpleNamespace(
    num_self_play_iterations=40, training_timesteps_per_role_training=100_000, archive_save_interval=1,
    policy_sample_strategy="pfsp", win_rate_buffer_size=20, n_trial_episodes=5,
    cop_role_prefix="cop", thief_role_prefix="thief")


# ------------------------------------------------------------------ win-rate table (policy_archive_utils.py:11-94)
def load_win_rates(role_archive_path: Path) -> dict:
    f = Path(role_archive_path) / WIN_RATES_FILENAME
    if not f.exists():
        return {}
    try:
        raw = json.loads(f.read_text())
    except json.JSONDecodeError:
        return {}
    for data in raw.values():
        size = data.get("buffer_size", 20)
        data["buffer_size"] = size
        if isinstance(data.get("recent_outcomes"), list):
            data["recent_outcomes"] = deque(data["recent_outcomes"], maxlen=size)
    return raw


def save_win_rates(role_archive_path: Path, win_rates_data: dict) -> None:
    out = {}
    for name, data in win_rates_data.items():
        d = dict(data)
        if isinstance(d.get("recent_outcomes"), deque):
            d["recent_outcomes"] = list(d["recent_outcomes"])
        out[name] = d
    Path(role_archive_path).mkdir(parents=True, exist_ok=True)
    (Path(role_archive_path) / WIN_RATES_FILENAME).write_text(json.dumps(out, indent=4))


def update_policy_win_rate(role_archive_path: Path, policy_filename: str, won_episode: bool, buffer_size: int) -> dict:
    data = load_win_rates(role_archive_path)
    st = data.setdefault(policy_filename, {"wins": 0, "games": 0, "recent_outcomes": deque(maxlen=buffer_size),
                                           "buffer_size": buffer_size})
    if st.get("buffer_size") != buffer_size or not isinstance(st["recent_outcomes"], deque):
        st["recent_outcomes"] = deque(list(st.get("recent_outcomes", [])), maxlen=buffer_size)
        st["buffer_size"] = buffer_size
    st["games"] += 1
    st["wins"] += 1 if won_episode else 0
    st["recent_outcomes"].append(1 if won_episode else 0)
    save_win_rates(role_archive_path, data)
    return st


# ------------------------------------------------------------------ archive (policy_archive_utils.py:97-127)
def add_policy_to_archive(checkpoint_path: str, role_archive_path: Path, iteration_number: int, role_prefix: str) -> Path:
    role_archive_path = Path(role_archive_path)
    role_archive_path.mkdir(parents=True, exist_ok=True)
    dst = role_archive_path / f"{role_prefix}_iter_{iteration_number}.pt"
    shutil.copy(checkpoint_path, dst)
    return dst


def _archived(role_archive_path: Path, role_prefix: str):
    p = Path(role_archive_path)
    return sorted(p.glob(f"{role_prefix}_iter_*.pt")) if p.exists() else []


def get_latest_policy_from_archive(role_archive_path: Path, role_prefix: str) -> Optional[str]:
    files = _archived(role_archive_path, role_prefix)
    return str(max(files, key=lambda q: int(q.stem.split("_")[-1]))) if files else None


def current_win_rate(stats: Optional[dict]) -> float:
    """Recent-window win rate if there is one, else lifetime, else 0.5 (policy_archive_utils.py:153-171)."""
    if not stats or stats.get("games", 0) <= 0:
        return DEFAULT_WIN_RATE
    recent = stats.get("recent_outcomes")
    if recent is not None and len(recent) > 0:
        return sum(recent) / len(recent)
    return stats["wins"] / stats["games"]


def pfsp_weight(win_rate: float) -> float:
    """Prioritised fictitious self-play: opponents near a 50 % win rate are sampled most (``:173-176``)."""
    return max(1e-3, 1.0 - abs(win_rate - 0.5) * 2.0)


def sample_policy_from_archive(role_archive_path: Path, role_prefix: str, strategy: str = "latest",
                               rng: Optional[random.Random] = None) -> Optional[str]:
    files = [str(q) for q in _archived(role_archive_path, role_prefix)]
    if not files:
        return None
    rng = rng or random
    if strategy == "random":
        return rng.choice(files)
    if strategy == "pfsp":
        table = load_win_rates(role_archive_path)
        weights = [pfsp_weight(current_win_rate(table.get(Path(f).name))) for f in files]
        return rng.choices(files, weights=weights, k=1)[0]
    return get_latest_policy_from_archive(role_archive_path, role_prefix)   # "latest" and unknown strategies


# ------------------------------------------------------------------ batched evaluation (eval_pfsp_agents.py:7-59)
def evaluate_agents(env, learner, n_episodes: int = 5, cop_prefix: str = "cop", thief_prefix: str = "thief",
                    greedy: bool = False, max_steps: Optional[int] = None, by_map: bool = False):
    """Play every world until it has finished ``n_episodes`` episodes with the learner's policies frozen;
    return (cop win rate, thief win rate) over all counted episodes.  The winner comes from the step kernel's
    ``winner`` output (0 cop, 1 thief), the batched form of ``infos[agent]["winner"]``.

    ``by_map=True`` (for a mixed-map environment) returns ``(cop rate, thief rate, per_map)`` instead, ``per_map``
    holding one dict per map of the environment — ``{"map", "cop", "thief", "episodes"}`` — from the episodes its
    worlds finished (``env.map_index``); their ``episodes`` add up to the episodes behind the overall rates."""
    import torch
    N, dev = env.num_envs, env.device
    limit = max_steps or (env.max_step_count + 1) * n_episodes
    finished = torch.zeros(N, dtype=torch.int32, device=dev)
    cop_wins = torch.zeros((), dtype=torch.int64, device=dev)
    thief_wins = torch.zeros((), dtype=torch.int64, device=dev)
    if by_map:
        map_index = getattr(env, "map_index", None)
        map_index = torch.zeros(N, dtype=torch.int64, device=dev) if map_index is None else map_index.to(dev, torch.int64)
        names = list(getattr(env, "map_names", None) or [f"map{m}" for m in range(int(map_index.max()) + 1)])
        cop_by_map = torch.zeros(len(names), dtype=torch.int64, device=dev)
        thief_by_map = torch.zeros(len(names), dtype=torch.int64, device=dev)
    was_training = {a: (learner.models[a]["policy"].training, learner.models[a]["value"].training) for a in learner.agents}
    for a in learner.agents:
        learner.models[a]["policy"].eval()
    learner.reset_recurrent_state()
    obs, _ = env.reset()
    with torch.no_grad():
        for _ in range(limit):
            actions = learner.act(obs, greedy=greedy)
            obs, _, term, _, infos = env.step(actions)
            done = term[learner.agents[0]].view(-1)
            winner = infos[learner.agents[0]]["winner"]
            counted = done & (finished < n_episodes)
            cop_wins += (counted & (winner == 0)).sum()
            thief_wins += (counted & (winner == 1)).sum()
            if by_map:
                cop_by_map += torch.bincount(map_index[counted & (winner == 0)], minlength=len(names))
                thief_by_map += torch.bincount(map_index[counted & (winner == 1)], minlength=len(names))
            finished += counted.to(torch.int32)
            learner.note_done(done)
            if bool((finished >= n_episodes).all()):
                break
    for a in learner.agents:
        learner.models[a]["policy"].train(was_training[a][0])
    learner.reset_recurrent_state()
    learner._obs = None          # the next rollout starts from a fresh reset, like env.reset() at eval_pfsp_agents.py:53
    total = max(int(finished.sum().item()), 1)
    if not by_map:
        return int(cop_wins.item()) / total, int(thief_wins.item()) / total
    episodes = torch.zeros(len(names), dtype=torch.int64, device=dev).index_add_(0, map_index, finished.to(torch.int64))
    per_map = []
    for m, name in enumerate(names):
        n_m = int(episodes[m].item())
        per_map.append({"map": name, "cop": int(cop_by_map[m].item()) / max(n_m, 1),
                        "thief": int(thief_by_map[m].item()) / max(n_m, 1), "episodes": n_m})
    return int(cop_wins.item()) / total, int(thief_wins.item()) / total, per_map


def evaluate_vs_scripted(env, learner, role_prefix: str, controller: str = "evade", n_episodes: int = 5,
                         by_map: bool = False, greedy: bool = False, cop_prefix: str = "cop", thief_prefix: str = "thief"):
    """Win rate of the learned role ``role_prefix`` against the step kernel's ``controller`` (``"evade"``, ``"chase"``
    or ``"random"``) playing every agent of the other role: a yardstick that does not move when the learner's own
    opponents change.  Needs ``BatchedCopsThievesEnv(scripted=...)``; the agents of ``role_prefix`` must have models in
    the learner.  The other role is scripted in every world, ``evaluate_agents`` runs (the kernel ignores the learner's
    actions for scripted agents), and the modes found are restored.  Returns the rate, or with ``by_map``
    ``(rate, [{"map", "rate", "episodes"} per map])``."""
    if role_prefix not in (cop_prefix, thief_prefix):
        raise ValueError(f"role_prefix must be {cop_prefix!r} or {thief_prefix!r}, got {role_prefix!r}")
    learned = [a for a in env.possible_agents if a.startswith(role_prefix)]
    missing = [a for a in learned if a not in learner.agents]
    if missing:
        raise ValueError(f"the learner has no models for {missing}")
    other = [a for a in env.possible_agents if not a.startswith(role_prefix)]
    w = env.worlds
    saved = w.script_modes.clone()
    try:
        env.set_scripted({a: controller for a in other})
        out = evaluate_agents(env, learner, n_episodes, cop_prefix, thief_prefix, greedy=greedy, by_map=by_map)
    finally:
        w.set_script_table(saved)
    key = "cop" if role_prefix == cop_prefix else "thief"
    rate = out[0] if key == "cop" else out[1]
    if not by_map:
        return rate
    return rate, [{"map": m["map"], "rate": m[key], "episodes": m["episodes"]} for m in out[2]]


def evaluate_agent(env, learner, learned_role_prefix: str, opponent_role_prefix: str, opponent_role_archive_path: Path,
                   training_config=TrainingConfig, num_additional_opponents_to_evaluate: int = 5,
                   rng: Optional[random.Random] = None) -> Dict[str, Tuple[float, float]]:
    """Evaluate the freshly trained role against up to N distinct archived opponents and update THEIR win
    rates (agent_learning_utils.py:233-380).  Returns {opponent file: (cop rate, thief rate)}."""
    results: Dict[str, Tuple[float, float]] = {}
    seen = set()
    keep = {a: {r: {k: v.clone() for k, v in learner.models[a][r].state_dict().items()} for r in ("policy", "value")}
            for a in learner.agents if a.startswith(opponent_role_prefix)}
    for _ in range(num_additional_opponents_to_evaluate):
        choice = None
        for strategy in (training_config.policy_sample_strategy, "random"):
            for _attempt in range(20):
                cand = sample_policy_from_archive(opponent_role_archive_path, opponent_role_prefix, strategy, rng)
                if cand is None:
                    break
                if Path(cand).name not in seen:
                    choice = cand
                    break
            if choice:
                break
        if not choice:
            break
        seen.add(Path(choice).name)
        learner.load(choice, role_prefix=opponent_role_prefix)          # copy_role_models for the opponent role
        cop_rate, thief_rate = evaluate_agents(env, learner, training_config.n_trial_episodes,
                                               training_config.cop_role_prefix, training_config.thief_role_prefix)
        opponent_won = thief_rate > cop_rate if learned_role_prefix == training_config.cop_role_prefix else cop_rate > thief_rate
        update_policy_win_rate(opponent_role_archive_path, Path(choice).name, opponent_won, training_config.win_rate_buffer_size)
        results[Path(choice).name] = (cop_rate, thief_rate)
    for a, roles in keep.items():                                        # put the trained opponent-role weights back
        for r, sd in roles.items():
            learner.models[a][r].load_state_dict(sd)
    return results


def self_play_iteration(env, learner, iteration: int, base_archive_path: Path, timesteps: int,
                        training_config=TrainingConfig, total_iterations: Optional[int] = None,
                        rng: Optional[random.Random] = None) -> str:
    """One pass of ``_orchestrate_simultaneous_training_iteration`` (orchestration.py:100-249): train both
    roles together for ``timesteps`` more lockstep steps, evaluate each role against the other role's archive,
    save ``joint_iter_{k}_full_agent.pt`` and archive it under both roles."""
    base = Path(base_archive_path)
    cop_dir, thief_dir = base / training_config.cop_role_prefix, base / training_config.thief_role_prefix
    base.mkdir(parents=True, exist_ok=True)
    learner.train(learner.timestep + timesteps)
    evaluate_agent(env, learner, training_config.cop_role_prefix, training_config.thief_role_prefix, thief_dir,
                   training_config, rng=rng)
    evaluate_agent(env, learner, training_config.thief_role_prefix, training_config.cop_role_prefix, cop_dir,
                   training_config, rng=rng)
    ckpt = base / f"joint_iter_{iteration}_full_agent.pt"
    learner.save(str(ckpt))
    total = total_iterations if total_iterations is not None else training_config.num_self_play_iterations
    if iteration % training_config.archive_save_interval == 0 or iteration == total - 1:
        add_policy_to_archive(str(ckpt), cop_dir, iteration, training_config.cop_role_prefix)
        add_policy_to_archive(str(ckpt), thief_dir, iteration, training_config.thief_role_prefix)
    return str(ckpt)
