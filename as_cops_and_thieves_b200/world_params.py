"""Per-world physics parameters (``cat_env_attach_world_params``): the table's layout, the ranges of domain
randomisation, and the checks of everything a caller writes into either.  Host only: nothing here needs a GPU.

Four parameters can differ between worlds, two of them also between the teams:

* ``unit_velocity`` — impulse of one action, per team (``[0]`` cops, ``[1]`` thieves), >= 0;
* ``max_speed`` — top speed, per team, > 0;
* ``termination_radius`` — capture radius, >= 0;
* ``max_step_count`` — time limit in steps, an integer >= 1.

A value for a team field is either one value for both teams or a dict by team name (``"cop"`` / ``"cops"``,
``"thief"`` / ``"thieves"``).  A range is a ``(lo, hi)`` pair, or one value to pin the field.
"""
from __future__ import annotations

import math
from typing import Dict, Iterator, Mapping, Optional, Sequence, Tuple, Union

import numpy as np

FIELDS = ("unit_velocity", "max_speed", "termination_radius", "max_step_count")
TEAM_FIELDS = ("unit_velocity", "max_speed")
TEAMS = {"cop": 0, "cops": 0, "thief": 1, "thieves": 1}

#: one entry of the per-world table (``CatWorldParams``, 24 bytes) and of the per-map-slot ranges (``CatWorldParamRanges``)
PARAMS_DTYPE = np.dtype([("unit_velocity", np.float32, 2), ("max_speed", np.float32, 2),
                         ("termination_radius", np.float32), ("max_step_count", np.int32)])
RANGES_DTYPE = np.dtype([("lo", PARAMS_DTYPE), ("hi", PARAMS_DTYPE), ("draw", np.int32)])
WORDS = PARAMS_DTYPE.itemsize // 4            # 6 four-byte words per world
RANGE_WORDS = RANGES_DTYPE.itemsize // 4      # 13 per map slot


def defaults(params: Mapping) -> np.ndarray:
    """The entry every world starts with: the environment's ``EnvParams`` values, the same for both teams (fp32, as the
    kernel reads them without a table)."""
    e = np.zeros((), PARAMS_DTYPE)
    e["unit_velocity"] = np.float32(params["unit_velocity"])
    e["max_speed"] = np.float32(params["max_speed"])
    e["termination_radius"] = np.float32(params["termination_radius"])
    e["max_step_count"] = int(params["max_step_count"])
    return e


def check_values(field: str, values) -> None:
    """Raise ``ValueError`` unless every value is allowed for ``field`` (numbers, numpy arrays or torch tensors)."""
    if field not in FIELDS:
        raise ValueError(f"unknown world parameter {field!r}; known: {', '.join(FIELDS)}")
    try:
        import torch
        if isinstance(values, torch.Tensor):
            values = values.detach().cpu().numpy()
    except ImportError:  # pragma: no cover
        pass
    a = np.asarray(values)
    if a.dtype == object or not (np.issubdtype(a.dtype, np.number) or a.dtype == bool):
        raise ValueError(f"{field}: values must be numbers")
    a = a.astype(np.float64)
    if not np.isfinite(a).all():
        raise ValueError(f"{field}: values must be finite")
    if field == "max_step_count":
        if (a != np.round(a)).any() or (a < 1).any() or (a > 2 ** 31 - 1).any():
            raise ValueError(f"{field}: the time limit must be an integer >= 1")
    elif field == "max_speed":
        if (a <= 0).any():
            raise ValueError(f"{field}: top speeds must be > 0")
    elif (a < 0).any():
        raise ValueError(f"{field}: values must be >= 0")


def per_team(field: str, value) -> Iterator[Tuple[Optional[int], object]]:
    """(team column or None, value) pairs of one assignment: a team field takes one value for both teams or a dict by
    team name; the other fields take one value."""
    if field not in FIELDS:
        raise ValueError(f"unknown world parameter {field!r}; known: {', '.join(FIELDS)}")
    if field not in TEAM_FIELDS:
        if isinstance(value, Mapping):
            raise ValueError(f"{field} is not a per-team parameter")
        yield None, value
    elif isinstance(value, Mapping):
        for team, v in value.items():
            if team not in TEAMS:
                raise ValueError(f"{field}: unknown team {team!r}; known: {', '.join(TEAMS)}")
            yield TEAMS[team], v
    else:
        yield 0, value
        yield 1, value


def _pair(field: str, r) -> Tuple[float, float]:
    if isinstance(r, (tuple, list)) and len(r) == 2:
        lo, hi = r
    elif isinstance(r, (tuple, list)):
        raise ValueError(f"{field}: a range is a (lo, hi) pair or one value, got {r!r}")
    else:
        lo = hi = r
    check_values(field, [lo, hi])
    if lo > hi:
        raise ValueError(f"{field}: lo {lo} > hi {hi}")
    return lo, hi


def ranges_entry(spec: Optional[Mapping], params: Mapping, draw: bool = True) -> np.ndarray:
    """One ``RANGES_DTYPE`` entry from a randomisation spec such as ``{"max_speed": {"thief": (125, 175)},
    "termination_radius": (15, 25), "max_step_count": (300, 500)}``: every field or team the spec does not name is
    pinned to the environment's value (``params``).  ``spec=None`` pins everything."""
    e = np.zeros((), RANGES_DTYPE)
    e["lo"] = e["hi"] = defaults(params)
    for field, r in (spec or {}).items():
        for col, v in per_team(field, r):
            lo, hi = _pair(field, v)
            if col is None:
                e["lo"][field], e["hi"][field] = lo, hi
            else:
                e["lo"][field][col], e["hi"][field][col] = lo, hi
    e["draw"] = 1 if draw else 0
    return e


def per_slot(spec: Union[None, Mapping, Sequence[Optional[Mapping]]], n_maps: int) -> list:
    """A spec for every map slot: one dict (or None) applies to all of them, a sequence gives one per slot."""
    if spec is None or isinstance(spec, Mapping):
        return [spec] * n_maps
    specs = list(spec)
    if len(specs) != n_maps:
        raise ValueError(f"one randomisation spec per map ({n_maps}), got {len(specs)}")
    return specs


def parse_cli(text: str) -> Dict:
    """``"max_speed.thief=125:175,termination_radius=15:25,max_step_count=400"`` -> a randomisation spec
    (``lo:hi`` a range, one number a pinned value, ``field.team`` one team of a per-team field)."""
    spec: Dict = {}
    for item in filter(None, (s.strip() for s in text.split(","))):
        key, sep, val = item.partition("=")
        if not sep:
            raise ValueError(f"--randomize item {item!r} is not field[.team]=lo:hi")
        field, _, team = key.strip().partition(".")
        num = (lambda s: int(s)) if field == "max_step_count" else float
        parts = val.split(":")
        try:
            r = (num(parts[0]), num(parts[1])) if len(parts) == 2 else num(parts[0])
        except (ValueError, IndexError):
            raise ValueError(f"--randomize item {item!r}: {val!r} is not lo:hi or one number") from None
        if len(parts) > 2 or (isinstance(r, float) and not math.isfinite(r)):
            raise ValueError(f"--randomize item {item!r}: {val!r} is not lo:hi or one number")
        if team:
            spec.setdefault(field, {})
            if not isinstance(spec[field], dict):
                raise ValueError(f"--randomize: {field} given for both teams and for one")
            spec[field][team] = r
        else:
            spec[field] = r
    for field, r in spec.items():
        for _, v in per_team(field, r):
            _pair(field, v)
    return spec
