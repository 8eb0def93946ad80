"""Scripted agents: the built-in controllers of the step kernel (``cat_env_attach_scripts``, include/cat_b200.h).

Each agent of each world has a mode, ``u8 mode[N][A]``: ``none`` (the caller's action), ``random``, ``chase`` or
``evade``.  Whenever a launch emits a world's observation, the kernel also writes what each controller would do next from
it into ``u8 decisions[N][A]`` (random in bits 0-1, chase in bits 2-3, evade in bits 4-5), and the next step acts on the
decision of every scripted agent instead of the caller's action.  This module holds the mode names and codes, the
checks the setters apply (the kernel validates nothing), and ``decode``.
"""
from __future__ import annotations

from typing import Dict, Mapping, Optional, Sequence, Union

import torch

from ._lib import CAT_SCRIPT_CHASE, CAT_SCRIPT_EVADE, CAT_SCRIPT_NONE, CAT_SCRIPT_RANDOM

#: mode name -> CAT_SCRIPT_* code
MODES: Dict[str, int] = {"none": CAT_SCRIPT_NONE, "random": CAT_SCRIPT_RANDOM, "chase": CAT_SCRIPT_CHASE,
                         "evade": CAT_SCRIPT_EVADE}
#: code -> mode name
NAMES: Dict[int, str] = {v: k for k, v in MODES.items()}

ModeLike = Union[str, int]


def mode_code(mode: ModeLike) -> int:
    """The CAT_SCRIPT_* code of a mode name (``"evade"``) or code (3); raises ValueError for anything else."""
    if isinstance(mode, str):
        if mode not in MODES:
            raise ValueError(f"unknown script mode {mode!r} (one of {', '.join(MODES)})")
        return MODES[mode]
    if isinstance(mode, bool) or not isinstance(mode, int) or mode not in NAMES:
        raise ValueError(f"script mode codes are 0..3, got {mode!r}")
    return int(mode)


def mode_name(code: int) -> str:
    """The name of a CAT_SCRIPT_* code."""
    return NAMES[mode_code(int(code))]


def check_modes(modes: torch.Tensor) -> None:
    """Every entry of an integer tensor of codes is in 0..3 (the kernel does not check the table)."""
    if modes.dtype.is_floating_point or modes.dtype == torch.bool:
        raise ValueError(f"script modes must be an integer tensor, got {modes.dtype}")
    if modes.numel() and (int(modes.min()) < 0 or int(modes.max()) > 3):
        raise ValueError("script mode codes are 0..3")


def check_mask(mask, n_worlds: int) -> torch.Tensor:
    """An (N,) bool mask of worlds on the CPU from a bool tensor, array or sequence; raises ValueError otherwise."""
    t = torch.as_tensor(mask)
    if t.dtype != torch.bool:
        raise ValueError(f"a world mask must be bool, got {t.dtype}")
    t = t.reshape(-1).cpu()
    if t.numel() != n_worlds:
        raise ValueError(f"mask needs {n_worlds} entries, got {t.numel()}")
    return t


def agent_modes(spec: Optional[Mapping], agents: Sequence[str]) -> Dict[int, int]:
    """``{agent name: mode}`` -> ``{agent index: code}`` against the environment's agent names, in index order."""
    out: Dict[int, int] = {}
    for name, mode in (spec or {}).items():
        if name not in agents:
            raise ValueError(f"unknown agent {name!r} (agents: {', '.join(agents)})")
        out[list(agents).index(name)] = mode_code(mode)
    return out


def parse_spec(text: str) -> Dict[str, str]:
    """``"thief_0=evade,cop_0=chase"`` -> ``{"thief_0": "evade", "cop_0": "chase"}`` (modes are checked)."""
    out: Dict[str, str] = {}
    for item in filter(None, (s.strip() for s in text.split(","))):
        name, sep, mode = item.partition("=")
        if not sep or not name.strip():
            raise ValueError(f"expected agent=mode, got {item!r}")
        mode_code(mode.strip())
        out[name.strip()] = mode.strip()
    return out


def decode(decisions: torch.Tensor, modes: torch.Tensor) -> torch.Tensor:
    """(N, A) int64 next actions of the scripted agents: ``(decisions >> 2 (mode - 1)) & 3`` where ``mode`` is
    non-zero, -1 where the agent is not scripted (its next action is the caller's)."""
    d = decisions.to(torch.int64)
    m = modes.to(torch.int64)
    act = (d >> (2 * (m - 1)).clamp(min=0)) & 3
    return torch.where(m > 0, act, torch.full_like(act, -1))
