"""``CatWorlds`` — N lockstep worlds on one GPU behind the C ABI (``include/cat_b200.h``).

Thin host object: owns the PyTorch tensors (packed state buffer + outputs), builds the
``CatStepIO`` pointer table once, and enqueues one kernel launch per ``reset`` / ``step`` /
``observe`` on the current torch CUDA stream.  No compute happens in Python and there is no CPU
path: constructing it without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import functools
from typing import Dict, Mapping, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib, episodes, scripts as cscripts, world_params as wparams
from ._lib import (CatEnvInfo, CatEpisodeStatsIO, CatScriptIO, CatWorldParamsIO, CatMapDesc, CatParams, CatRecordLayout, CatStateView, CatStepIO,
                   CAT_WALL_SLOTS)
from .maps import CompiledMap
from .params import EnvParams

ActionsLike = Union[torch.Tensor, Mapping[str, torch.Tensor], Sequence[torch.Tensor]]


def _require_cuda(device: torch.device) -> None:
    if device.type != "cuda" or not torch.cuda.is_available():
        raise _lib.CatError(
            "as_cops_and_thieves_b200 needs a CUDA device (sm_100a); there is no CPU fallback "
            f"(requested device={device}, torch.cuda.is_available()={torch.cuda.is_available()})")


class HostRecords(dict):
    """What ``CatWorlds.step_host`` returns: views of the pinned host record buffer.  With packed records ``obs_type`` is
    not a view — it is decoded from ``obs_type_packed`` when asked for (and not cached: the buffer is rewritten by the
    next call)."""
    shape = (0, 0)

    def __missing__(self, key):
        if key == "obs_type" and "obs_type_packed" in self:
            return CatWorlds.unpack_types(self["obs_type_packed"], *self.shape)
        raise KeyError(key)


def _map_desc(cmap: CompiledMap):
    """``CatMapDesc`` of a compiled map, and the numpy arrays it points into (keep them alive while it is used)."""
    keep = dict(
        hull_off=np.ascontiguousarray(cmap.hull_off, np.int32),
        vert=np.ascontiguousarray(cmap.vert, np.float64),
        normal=np.ascontiguousarray(cmap.normal, np.float64),
        edge_len=np.ascontiguousarray(cmap.edge_len, np.float64),
        hull_bb=np.ascontiguousarray(cmap.hull_bb, np.float64),
        init_pos=np.ascontiguousarray(cmap.init_pos, np.float64),
        region_off=np.ascontiguousarray(cmap.region_off, np.int32),
        regions=np.ascontiguousarray(cmap.regions if len(cmap.regions) else np.zeros((1, 4)), np.float64),
        con_cell_off=np.ascontiguousarray(cmap.con_cell_off, np.int32),
        con_cell_hulls=np.ascontiguousarray(np.append(cmap.con_cell_hulls, 0), np.int32),
        view_cell_off=np.ascontiguousarray(cmap.view_cell_off, np.int32),
        view_cell_edges=np.ascontiguousarray(np.append(cmap.view_cell_edges, 0), np.int32),
    )
    k = keep
    md = CatMapDesc(
        cmap.n_hulls, cmap.n_edges, _lib.np_ptr(k["hull_off"]), _lib.np_ptr(k["vert"]), _lib.np_ptr(k["normal"]),
        _lib.np_ptr(k["edge_len"]), _lib.np_ptr(k["hull_bb"]), cmap.n_cops, cmap.n_thieves,
        _lib.np_ptr(k["init_pos"]), _lib.np_ptr(k["region_off"]), _lib.np_ptr(k["regions"]),
        cmap.grid_x0, cmap.grid_y0, cmap.cell, cmap.nx, cmap.ny,
        _lib.np_ptr(k["con_cell_off"]), _lib.np_ptr(k["con_cell_hulls"]),
        _lib.np_ptr(k["view_cell_off"]) if len(k["view_cell_off"]) == cmap.nx * cmap.ny + 1 else None,
        _lib.np_ptr(k["view_cell_edges"]), float(cmap.view_range))
    return md, keep


def _cat_params(p: Mapping) -> CatParams:
    return CatParams(**{name: p[name] for name, _ in CatParams._fields_})


def map_blob_bytes(cmap: CompiledMap, params: Mapping) -> int:
    """``cat_map_blob_bytes``: the shared-memory blob of ``cmap`` under the parameters ``params`` (an ``EnvParams``
    dict), what a swappable environment's ``map_blob_capacity`` must cover.  Host only."""
    L = _lib.load()
    md, _keep = _map_desc(cmap)
    cp = _cat_params(params)
    out = C.c_int32(0)
    _lib.check(L.cat_map_blob_bytes(C.byref(md), C.byref(cp), C.byref(out)), "cat_map_blob_bytes")
    return int(out.value)


@functools.lru_cache(maxsize=8)
def _shipped_blob_capacity(key: tuple) -> int:
    from .maps import SHIPPED_MAPS, compile_map, free_space_regions, load_named_map
    params = dict(key)
    best = 0
    for name in SHIPPED_MAPS:
        m = load_named_map(name)
        for so in (None, free_space_regions(m)):
            best = max(best, map_blob_bytes(compile_map(m, name=name, spawn_override=so), params))
    return best


def default_blob_capacity(params: Mapping) -> int:
    """The largest blob of the shipped maps (with their own spawn regions and with ``free_space_regions``) under
    ``params``: the default ``map_blob_capacity`` of a swappable environment (agh-map's blob)."""
    return _shipped_blob_capacity(tuple(sorted((k, params[k]) for k, _ in CatParams._fields_)))


class CatWorlds:
    def __init__(self, cmap: Union[CompiledMap, Sequence[CompiledMap]], n_worlds: Union[int, Sequence[int]], *,
                 device: Union[str, torch.device] = "cuda:0",
                 gid0: int = 0, params: Optional[EnvParams] = None, want_f32: bool = True,
                 want_shared: bool = True, want_hits: bool = False, pinned_outputs: bool = False,
                 want_critic: bool = False, want_bf16: bool = False, want_final: bool = False,
                 swappable_maps: bool = False, map_blob_capacity: Optional[int] = None,
                 want_episode_stats: bool = False, want_world_params: bool = False,
                 param_ranges: Union[None, Mapping, Sequence[Optional[Mapping]]] = None,
                 want_scripts: bool = False, scripts: Optional[Mapping[int, Union[str, int]]] = None, **overrides):
        """``pinned_outputs=True`` places every output tensor in mapped pinned HOST memory: the kernel stores its
        results there directly and the host reads them (``tensor.numpy()``) after one stream synchronisation —
        the layout for callers that consume every step on the CPU, like the single-world PettingZoo face.
        ``want_critic``: also emit the critic's 4-channel ray block ``critic_f32 (N, 4, R)``
        (``lstm_value_net.py:122-137``); ``want_bf16``: bf16 copies of ``obs_f32`` / ``critic_f32``.

        ``want_final``: every step also writes, for each world that ENDS in it (``terminated``), what the step would
        have emitted with ``auto_reset = 0`` — the observation of the positions it ended in with the terminal rewards
        and flags — into a second set of outputs: the record views ``final_obs_dist``, ``final_obs_type``,
        ``final_reward``, ``final_terminated``, ``final_truncated``, ``final_winner``, and ``final_obs_f32`` /
        ``final_state_f32`` / ``final_critic_f32`` where ``want_f32`` / ``want_critic`` ask for the plain ones.  With
        auto-reset the plain outputs of such a world already hold the new episode, so this is the only copy of its last
        observation (gymnasium's ``final_observation``).  Entries of worlds that do not end are left untouched: read them
        where ``terminated``.

        Mixed maps: ``cmap`` may be a sequence of compiled maps (at most ``CAT_MAX_MAPS``, all with the same cops and
        thieves) with ``n_worlds`` the matching sequence of world counts.  Map m then owns the worlds
        ``world_offsets[m] .. world_offsets[m] + n_worlds[m]`` and all of them are stepped by one launch; world i is
        the same world as world ``i - world_offsets[m]`` of a single-map ``CatWorlds`` of map m with
        ``gid0 + world_offsets[m]``.  ``cmaps``, ``world_offsets`` and ``map_index`` (the map of every world, (N,) int64
        on the device) describe the split; with one map they hold that map alone.

        ``swappable_maps``: the environment is created by ``cat_env_create_swappable``, so ``set_map`` can replace any
        of its maps later without invalidating its buffers or a captured CUDA graph.  Each map's blob is then allocated
        at ``map_blob_capacity`` bytes (a positive multiple of 16; default: the largest blob of the creation maps and the
        shipped maps, ``default_blob_capacity``), and the mixed-map kernels run even for one map.  Needs ray lists
        (``ray_list_cell >= 0``).

        ``want_episode_stats``: the step kernel keeps each world's running return ``episode_acc`` (N, A) and, for every
        world that ends in a step, writes that episode's return ``episode_return`` (N, A) float32 and length
        ``episode_length`` (N,) int32 (valid where ``terminated``) and adds it to its map slot's totals, read with
        ``episode_totals`` (``cat_env_attach_episode_stats``; resets zero the running returns and never count an
        episode).  A step stays one launch; it runs the full-output kernel.

        ``want_world_params``: every world reads its thrust and top speed per team, its capture radius and its time limit
        from a device table (``cat_env_attach_world_params``), filled with this environment's values for both teams;
        ``world_params()`` gives named views of it and ``set_world_params`` writes it.  ``param_ranges`` (implies
        ``want_world_params``): a randomisation spec for every map slot, or one per slot (``set_param_ranges``), from
        which every re-spawn of a world draws its next entry.  A step stays one launch; it runs the full-output kernel.

        ``want_scripts``: built-in controllers can act for chosen agents inside the step kernel (``cat_env_attach_scripts``,
        ``scripts.py``): ``script_modes`` (N, A) uint8 holds each agent's mode (0 none, 1 random, 2 chase, 3 evade),
        written with ``set_scripts``, and ``script_decisions`` (N, A) uint8 what the controllers decided from the last
        emitted observation.  ``scripts`` (implies ``want_scripts``): initial ``{agent index: mode}`` for every world.
        A step stays one launch; it runs the full-output kernel."""
        if map_blob_capacity is not None and (int(map_blob_capacity) < 16 or int(map_blob_capacity) % 16):
            # the step kernel stages a blob with one bulk copy whose size must be a multiple of 16 bytes
            raise ValueError(f"map_blob_capacity must be a positive multiple of 16, got {map_blob_capacity}")
        if isinstance(cmap, CompiledMap):
            multi, cmaps, counts = False, [cmap], [int(n_worlds)]
        else:
            multi, cmaps = True, list(cmap)
            if isinstance(n_worlds, (int, np.integer)):
                raise ValueError("with a sequence of maps, n_worlds is the sequence of their world counts")
            counts = [int(n) for n in n_worlds]
            if len(counts) != len(cmaps) or not cmaps:
                raise ValueError(f"{len(cmaps)} maps need as many world counts, got {len(counts)}")
        self.device = torch.device(device)
        _require_cuda(self.device)
        self.L = _lib.load()
        self.cmaps = cmaps
        self.cmap = cmaps[0]
        self.worlds_per_map = tuple(counts)
        self.world_offsets = tuple(int(v) for v in np.cumsum([0] + counts[:-1]))
        p = (params or EnvParams()).as_dict()
        p.update(overrides)
        self.params = p
        self.n_worlds = int(sum(counts))
        self.gid0 = int(gid0)

        descs = [_map_desc(m) for m in cmaps]
        self._keep = [kp for _, kp in descs]
        cp = _cat_params(p)
        handle = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.swappable = bool(swappable_maps)
        self.maps_replaced = 0       # set_map calls so far (render.TrajectoryRecorder checks it)
        if self.swappable:
            if map_blob_capacity is None:
                map_blob_capacity = max([default_blob_capacity(p)] + [map_blob_bytes(m, p) for m in cmaps])
            self.map_blob_capacity = int(map_blob_capacity)
            mds = (CatMapDesc * len(cmaps))(*[md for md, _ in descs])
            cnt = (C.c_int32 * len(counts))(*counts)
            _lib.check(self.L.cat_env_create_swappable(mds, len(cmaps), cnt, C.byref(cp), self.map_blob_capacity, self.gid0,
                                                       dev_index, C.byref(handle)), "cat_env_create_swappable")
        elif multi:
            mds = (CatMapDesc * len(cmaps))(*[md for md, _ in descs])
            cnt = (C.c_int32 * len(counts))(*counts)
            _lib.check(self.L.cat_env_create_multi(mds, len(cmaps), cnt, C.byref(cp), self.gid0, dev_index,
                                                   C.byref(handle)), "cat_env_create_multi")
        else:
            _lib.check(self.L.cat_env_create(C.byref(descs[0][0]), C.byref(cp), self.n_worlds, self.gid0, dev_index,
                                             C.byref(handle)), "cat_env_create")
        self._h = handle
        info = CatEnvInfo()
        _lib.check(self.L.cat_env_info(self._h, C.byref(info)), "cat_env_info")
        self.info = info
        self.A, self.R, self.S, self.P = info.n_agents, info.n_rays, info.state_dim, info.n_pairs
        self.n_cops, self.n_thieves = info.n_cops, info.n_thieves
        self.map_index = torch.repeat_interleave(torch.arange(len(cmaps), dtype=torch.int64),
                                                 torch.tensor(counts, dtype=torch.int64)).to(self.device)

        N, A, R, dev = self.n_worlds, self.A, self.R, self.device
        nbytes = int(self.L.cat_env_state_bytes(self._h))
        self.state = torch.zeros(nbytes, dtype=torch.uint8, device=dev)   # packed per-world records
        # The per-step results are ONE record per world (include/cat_b200.h CatRecordLayout):
        #   [f16 distance A*R | u8 type A*R | f32 reward A | u8 terminated | u8 truncated | i8 winner], 16-byte aligned,
        # written by the kernel with 16-byte stores; the tensors below are strided views of the record buffer, so the
        # host-facing path moves any range of worlds with a single copy.
        rl = CatRecordLayout()
        _lib.check(self.L.cat_env_record_layout(self._h, C.byref(rl)), "cat_env_record_layout")
        self.record_layout = rl
        self.record_bytes = int(rl.bytes)
        # the host-facing form of the same record: types packed to 2 bits each (what step_host moves over PCIe by default)
        rp = CatRecordLayout()
        _lib.check(self.L.cat_env_packed_record_layout(self._h, C.byref(rp)), "cat_env_packed_record_layout")
        self.packed_record_layout = rp
        self.packed_record_bytes = int(rp.bytes)
        self.pinned_outputs = bool(pinned_outputs)

        def alloc(shape, dtype):
            if self.pinned_outputs:
                return torch.zeros(shape, dtype=dtype).pin_memory()
            return torch.zeros(shape, dtype=dtype, device=dev)
        self._out = alloc(N * self.record_bytes, torch.uint8)
        views = self._record_views(self._out)
        self.obs_dist, self.obs_type, self.reward = views["obs_dist"], views["obs_type"], views["reward"]
        self.terminated, self.truncated, self.winner = views["terminated"], views["truncated"], views["winner"]
        self.winner.fill_(-1)
        self.shared_dist = alloc((N, 2, R), torch.float16) if want_shared else None
        self.shared_type = alloc((N, 2, R), torch.uint8) if want_shared else None
        self.team_pos = alloc((N, A, 2), torch.float16) if want_shared else None
        self.obs_f32 = alloc((A, N, 2 * R), torch.float32) if want_f32 else None
        self.state_f32 = alloc((N, self.S), torch.float32) if want_f32 else None
        self.hit_point = alloc((N, A, R, 2), torch.float32) if want_hits else None
        self.critic_f32 = alloc((N, 4, R), torch.float32) if want_critic else None
        self.obs_bf16 = alloc((A, N, 2 * R), torch.bfloat16) if want_bf16 and want_f32 else None
        self.critic_bf16 = alloc((N, 4, R), torch.bfloat16) if want_bf16 and want_critic else None
        self.want_final = bool(want_final)
        self._final_out = alloc(N * self.record_bytes, torch.uint8) if want_final else None
        fviews = self._record_views(self._final_out) if want_final else dict.fromkeys(views)
        self.final_obs_dist, self.final_obs_type, self.final_reward = fviews["obs_dist"], fviews["obs_type"], fviews["reward"]
        self.final_terminated, self.final_truncated = fviews["terminated"], fviews["truncated"]
        self.final_winner = fviews["winner"]
        if want_final:
            self.final_winner.fill_(-1)
        self.final_obs_f32 = alloc((A, N, 2 * R), torch.float32) if want_final and want_f32 else None
        self.final_state_f32 = alloc((N, self.S), torch.float32) if want_final and want_f32 else None
        self.final_critic_f32 = alloc((N, 4, R), torch.float32) if want_final and want_critic else None
        self._host = None
        self._io = self._make_io()
        self._ptr_table = (C.c_void_p * 8)()
        self.want_episode_stats = bool(want_episode_stats)
        self.episode_acc = self.episode_return = self.episode_length = self._episode_totals = None
        if want_episode_stats:
            # always device memory: the kernel updates the totals with atomics
            self.episode_acc = torch.zeros((N, A), dtype=torch.float32, device=dev)
            self.episode_return = torch.zeros((N, A), dtype=torch.float32, device=dev)
            self.episode_length = torch.zeros(N, dtype=torch.int32, device=dev)
            self._episode_totals = torch.zeros(len(cmaps) * episodes.TOTALS_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            sio = CatEpisodeStatsIO(self.episode_acc.data_ptr(), self.episode_return.data_ptr(),
                                    self.episode_length.data_ptr(), self._episode_totals.data_ptr())
            _lib.check(self.L.cat_env_attach_episode_stats(self._h, C.byref(sio)), "cat_env_attach_episode_stats")
        self.want_world_params = bool(want_world_params) or param_ranges is not None
        self._wp = self._wp_ranges = None
        if self.want_world_params:
            # [N] CatWorldParams and [n_maps] CatWorldParamRanges as 4-byte words, read and written in place
            self._wp = torch.from_numpy(np.tile(wparams.defaults(p), N).view(np.int32).reshape(N, wparams.WORDS)).to(dev)
            self._ranges_host = np.zeros(len(cmaps), wparams.RANGES_DTYPE)
            self._ranges_host[:] = wparams.ranges_entry(None, p, draw=False)
            self._wp_ranges = torch.zeros((len(cmaps), wparams.RANGE_WORDS), dtype=torch.int32, device=dev)
            for slot, spec in enumerate(wparams.per_slot(param_ranges, len(cmaps))):
                if spec is not None:
                    self._ranges_host[slot] = wparams.ranges_entry(spec, p)
            self._upload_ranges()
            wio = CatWorldParamsIO(self._wp.data_ptr(), self._wp_ranges.data_ptr())
            _lib.check(self.L.cat_env_attach_world_params(self._h, C.byref(wio)), "cat_env_attach_world_params")
        self.want_scripts = bool(want_scripts) or scripts is not None
        self._script_mode = self._script_dec = self._script_mode_host = None
        if self.want_scripts:
            self._script_mode = torch.zeros((N, A), dtype=torch.uint8, device=dev)
            self._script_dec = torch.zeros((N, A), dtype=torch.uint8, device=dev)
            self._script_mode_host = np.zeros((N, A), np.uint8)   # mirror of the modes, kept by set_scripts
            if scripts:
                self.set_scripts(scripts)
            scio = CatScriptIO(self._script_mode.data_ptr(), self._script_dec.data_ptr())
            _lib.check(self.L.cat_env_attach_scripts(self._h, C.byref(scio)), "cat_env_attach_scripts")
        _lib.check(self.L.cat_env_init_state(self._h, self.state.data_ptr(), self._stream()), "cat_env_init_state")

    # ------------------------------------------------------------------ plumbing
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _record_views(self, buf: torch.Tensor, packed: bool = False) -> Dict[str, torch.Tensor]:
        """Strided tensor views of a record buffer (``N * record_bytes`` uint8, device or pinned host).  ``packed``: the
        buffer holds the packed form — ``obs_type_packed`` (N, ceil(A R / 4)) uint8 instead of ``obs_type``."""
        N, A, R = self.n_worlds, self.A, self.R
        rl = self.packed_record_layout if packed else self.record_layout
        rb = int(rl.bytes)
        f16, f32 = buf.view(torch.float16), buf.view(torch.float32)
        views = dict(
            obs_dist=f16.as_strided((N, A, R), (rb // 2, R, 1), rl.off_dist // 2),
            reward=f32.as_strided((N, A), (rb // 4, 1), rl.off_reward // 4),
            terminated=buf.as_strided((N,), (rb,), rl.off_terminated),
            truncated=buf.as_strided((N,), (rb,), rl.off_truncated),
            winner=buf.view(torch.int8).as_strided((N,), (rb,), rl.off_winner))
        if packed:
            views["obs_type_packed"] = buf.as_strided((N, (A * R + 3) // 4), (rb, 1), rl.off_type)
        else:
            views["obs_type"] = buf.as_strided((N, A, R), (rb, R, 1), rl.off_type)
        return views

    @staticmethod
    def unpack_types(packed: torch.Tensor, A: int, R: int) -> torch.Tensor:
        """(N, ceil(A R / 4)) uint8 of a packed record -> (N, A, R) uint8 ObjectType values (CatRecordLayout: ray r is
        bits 2 (r % 4) .. + 1 of byte r // 4; code 3 = EMPTY = 4)."""
        shifts = torch.tensor([0, 2, 4, 6], dtype=torch.uint8, device=packed.device)
        codes = ((packed.unsqueeze(-1) >> shifts) & 3).reshape(packed.shape[0], -1)[:, :A * R]
        return (codes + (codes == 3).to(torch.uint8)).reshape(packed.shape[0], A, R)

    def _make_io(self, record: Optional[torch.Tensor] = None, extras: bool = True, packed: bool = False) -> CatStepIO:
        def dp(t):
            return None if t is None or not extras else t.data_ptr()
        rec = self._out if record is None else record
        return CatStepIO(shared_dist=dp(self.shared_dist), shared_type=dp(self.shared_type), team_pos=dp(self.team_pos),
                         obs_f32=dp(self.obs_f32), state_f32=dp(self.state_f32), hit_point=dp(self.hit_point),
                         record=rec.data_ptr(), record_world_stride=self.packed_record_bytes if packed else self.record_bytes,
                         critic_f32=dp(self.critic_f32), obs_bf16=dp(self.obs_bf16), critic_bf16=dp(self.critic_bf16),
                         record_packed_types=1 if packed else 0, final_record=dp(self._final_out),
                         final_record_world_stride=self.record_bytes, final_obs_f32=dp(self.final_obs_f32),
                         final_state_f32=dp(self.final_state_f32), final_critic_f32=dp(self.final_critic_f32))

    def map_info(self, m: int) -> CatEnvInfo:
        """``cat_env_map_info``: the figures of map ``m`` alone (its worlds, hulls, edges, blob and ray-list bytes)."""
        info = CatEnvInfo()
        _lib.check(self.L.cat_env_map_info(self._h, int(m), C.byref(info)), "cat_env_map_info")
        return info

    def set_map(self, m: int, cmap: CompiledMap) -> torch.Tensor:
        """Replace map ``m`` of a swappable environment by ``cmap`` (same cops and thieves; its blob must fit
        ``map_blob_capacity``) and reset that map's worlds: ``cat_env_set_map``, then ``reset(mask)``, so the outputs of
        those worlds hold their first observation on the new map, as after ``reset(mask)``.  The other worlds are not
        touched.  Synchronises the device and may allocate: call it between steps, outside graph capture.  A CUDA graph
        captured before stays valid and steps the new map on its next replay.  Returns the (N,) bool mask of the reset
        worlds (a recurrent learner zeroes their states: ``MAPPOLearner.note_reset``).  On failure nothing changes."""
        m = int(m)
        if not 0 <= m < len(self.cmaps):
            raise IndexError(f"map index {m} out of range (0..{len(self.cmaps) - 1})")
        md, keep = _map_desc(cmap)
        _lib.check(self.L.cat_env_set_map(self._h, m, C.byref(md), self._stream()), "cat_env_set_map")
        del keep
        self.cmaps[m] = cmap
        self.cmap = self.cmaps[0]
        self.maps_replaced += 1
        info = CatEnvInfo()
        _lib.check(self.L.cat_env_info(self._h, C.byref(info)), "cat_env_info")
        self.info = info
        if getattr(self, "_renderer", None) is not None:   # it holds the old map's wall layer: rebuilt on next use
            self._renderer.close()
            self._renderer = None
        mask = self.map_index == m
        self.reset(mask)
        return mask

    def overflow_counts(self, reset: bool = False):
        """(wall contacts beyond CAT_WALL_SLOTS, near hulls beyond CAT_NEAR_SLOTS) since creation / the last reset
        of the counters — the fixed capacities the reference does not have; zero means they never mattered."""
        out = (C.c_uint64 * 2)()
        _lib.check(self.L.cat_env_overflow_counts(self._h, C.byref(out), int(reset)), "cat_env_overflow_counts")
        return int(out[0]), int(out[1])

    def close(self) -> None:
        if getattr(self, "_renderer", None) is not None:
            self._renderer.close()
            self._renderer = None
        if getattr(self, "_h", None):
            self.L.cat_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_seed(self, seed: int, restart_episodes: bool = False) -> None:
        """Re-key the spawn RNG.  ``restart_episodes`` also zeroes the per-world episode counters (part of the RNG
        key), so that ``reset(seed=s)`` reproduces the same spawns every time, like re-creating the reference's
        ``np_random`` (``base_env.py:307-311``)."""
        _lib.check(self.L.cat_env_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF), "cat_env_set_seed")
        self.params["seed"] = int(seed)
        if restart_episodes:
            self.set_state(episode=torch.zeros(self.n_worlds, dtype=torch.int32))

    # ------------------------------------------------------------------ the three launches
    def reset(self, mask: Optional[torch.Tensor] = None) -> None:
        """``BaseEnv.reset`` for the masked worlds (all if ``mask`` is None); fills the obs outputs."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            assert mask.numel() == self.n_worlds
        self._io.reset_mask = None if mask is None else mask.data_ptr()
        _lib.check(self.L.cat_env_reset(self._h, self.state.data_ptr(), C.byref(self._io), self._stream()),
                   "cat_env_reset")
        self._io.reset_mask = None

    def step(self, actions: ActionsLike) -> None:
        """``BaseEnv.step`` for every world: one kernel launch on the current stream."""
        io = self._io
        if isinstance(actions, torch.Tensor):
            on_device = actions.device == self.device or (actions.device.type == "cpu" and actions.is_pinned())
            if not on_device or not actions.is_contiguous() or actions.numel() != self.n_worlds * self.A:
                raise ValueError("actions must be a contiguous (N, A) tensor on the env's device (or in pinned host memory)")
            kind = {torch.uint8: 0, torch.int32: 1, torch.int64: 2}.get(actions.dtype)
            if kind is None:
                raise ValueError(f"unsupported action dtype {actions.dtype}")
            io.actions, io.actions_kind = actions.data_ptr(), kind
        else:
            seq = list(actions.values()) if isinstance(actions, Mapping) else list(actions)
            if len(seq) != self.A:
                raise ValueError(f"need {self.A} per-agent action tensors")
            for a, t in enumerate(seq):
                if t.dtype != torch.int64 or t.device != self.device or not t.is_contiguous() or t.numel() != self.n_worlds:
                    raise ValueError("per-agent actions must be contiguous int64 tensors of N elements on the env's device")
                self._ptr_table[a] = t.data_ptr()
            io.actions, io.actions_kind = C.cast(self._ptr_table, C.c_void_p), 3
        _lib.check(self.L.cat_env_step(self._h, self.state.data_ptr(), C.byref(io), self._stream()), "cat_env_step")

    # ------------------------------------------------------------------ host-buffer face (what a CPU caller sees)
    @property
    def h2d_bytes_per_step(self) -> int:
        return self.n_worlds * self.A

    @property
    def d2h_bytes_per_step(self) -> int:
        """Bytes that cross to the host per ``step_host`` in its default (packed) form."""
        return self.d2h_bytes(True)

    def d2h_bytes(self, packed: bool = True) -> int:
        """One output record per world (observations, rewards, flags and the record's alignment padding): 640 B packed
        (types at 2 bits), 832 B with u8 types, for 3 agents x 90 rays."""
        return self.n_worlds * (self.packed_record_bytes if packed else self.record_bytes)

    def _host_buffers(self, packed: bool = True) -> "HostRecords":
        """Pinned host record buffer, its strided views, and the I/O table that points the kernel straight at it (pinned
        memory is mapped into the device's address space); for the packed form also a device staging buffer of that
        layout for the DMA strategies (the device-resident ``self._out`` keeps u8 types for device consumers)."""
        if self._host is None:
            self._host = {}
        if packed not in self._host:
            if self.pinned_outputs:
                raise _lib.CatError("step_host needs device-resident outputs (pinned_outputs=False)")
            N, A = self.n_worlds, self.A
            rb = self.packed_record_bytes if packed else self.record_bytes
            hb = torch.zeros(N * rb, dtype=torch.uint8).pin_memory()
            h = HostRecords(blob=hb, actions_dev=torch.zeros((N, A), dtype=torch.uint8, device=self.device),
                            actions_pinned=torch.zeros((N, A), dtype=torch.uint8).pin_memory(), **self._record_views(hb, packed))
            h.shape = (A, self.R)
            h["record_bytes"] = rb
            h["io"] = self._make_io(record=hb, extras=False, packed=packed)
            h["dev"] = torch.zeros(N * rb, dtype=torch.uint8, device=self.device) if packed else self._out
            h["io_dev"] = self._make_io(record=h["dev"], extras=False, packed=packed)
            self._host[packed] = h
        return self._host[packed]

    def default_chunks(self) -> int:
        """Chunks for the pipelined host path: each chunk is one launch + one DMA copy of its records, the copy of
        chunk i overlapping the launch of chunk i + 1 (measured on B200, profiles/r2_notes.md)."""
        return 4 if self.n_worlds >= 2048 else 1

    def step_host(self, host_actions: torch.Tensor, mode: str = "auto", chunks: Optional[int] = None,
                  packed: bool = True) -> "HostRecords":
        """``step`` for a caller whose buffers live in host memory (the reference's own calling convention):
        uint8 actions ``(N, A)`` in, and the step's observations, rewards and flags in pinned host memory
        when the call returns (strided views of one record buffer: ``obs_dist`` f16, ``reward``, ``terminated``,
        ``truncated``, ``winner``, and the types).

        ``packed`` (default): the records cross PCIe in their packed form — ray types at 2 bits each, 640 B instead of
        832 B per world; the result holds ``obs_type_packed`` (a view) and decodes ``obs_type`` (N, A, R) uint8 on first
        access (``unpack_types``, a host-side bit unpack).  ``packed=False`` moves u8 types (``obs_type`` is a view).

        Three ways to move the results, same bytes, same values:

        * ``"pipelined"`` — ``cat_env_step_host``: the worlds are stepped in ``chunks`` launches; each
          chunk's block of records is DMA-copied with ONE ``cudaMemcpyAsync`` on a second stream while the next
          chunk computes; the kernel reads the actions straight from the pinned buffer.
        * ``"zero_copy"`` — one launch whose 16-byte stores go straight into mapped pinned host memory, so the
          transfer of one world's results overlaps the computation of the others (SM-issued PCIe writes).
        * ``"staged"`` — H2D copy, one launch, one D2H copy of the record buffer, strictly in sequence.

        ``"auto"`` (default) times the three on this environment's first calls (each trial is a real step) and keeps
        the fastest: which one wins depends on the step's length and on how many GPUs share the host's PCIe root
        (profiles/r2_notes.md: the SM-issued stores of zero-copy sustain 32-39 GB/s, a DMA copy 52 GB/s but a chunk's
        launch lasts a whole single-wave step).
        """
        if mode == "auto":
            mode = self._auto_mode(packed)
            if mode is None:
                return self._auto_trial(host_actions, packed)
        if mode not in ("pipelined", "zero_copy", "staged"):
            raise ValueError(f"unknown step_host mode {mode!r}")
        h = self._host_buffers(packed)
        if mode != "staged":
            if not host_actions.is_pinned():
                h["actions_pinned"].copy_(host_actions)
                host_actions = h["actions_pinned"]
            if host_actions.dtype != torch.uint8 or not host_actions.is_contiguous() or host_actions.numel() != self.n_worlds * self.A:
                raise ValueError("host actions must be a contiguous uint8 (N, A) tensor")
            if mode == "zero_copy":
                io = h["io"]
                io.actions, io.actions_kind = host_actions.data_ptr(), 0
                _lib.check(self.L.cat_env_step(self._h, self.state.data_ptr(), C.byref(io), self._stream()), "cat_env_step")
            else:
                _lib.check(self.L.cat_env_step_host(self._h, self.state.data_ptr(), host_actions.data_ptr(),
                                                    h["dev"].data_ptr(), h["blob"].data_ptr(), h["record_bytes"],
                                                    1 if packed else 0, int(chunks or self.default_chunks()),
                                                    self._stream()), "cat_env_step_host")
        else:
            h["actions_dev"].copy_(host_actions, non_blocking=True)
            io = h["io_dev"]
            io.actions, io.actions_kind = h["actions_dev"].data_ptr(), 0
            _lib.check(self.L.cat_env_step(self._h, self.state.data_ptr(), C.byref(io), self._stream()), "cat_env_step")
            h["blob"].copy_(h["dev"], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return h

    _AUTO_ORDER = ("zero_copy", "pipelined", "staged")
    _AUTO_TRIALS = 4           # timed calls per mode (after one untimed call each)

    def _auto_mode(self, packed: bool = True) -> Optional[str]:
        return getattr(self, "_auto_choices", {}).get(packed)

    @property
    def _auto_choice(self) -> Optional[str]:
        return self._auto_mode(True)

    def _auto_trial(self, host_actions: torch.Tensor, packed: bool = True) -> "HostRecords":
        import time
        states = self.__dict__.setdefault("_auto_state", {})
        st = states.setdefault(packed, {"i": 0, "t": {m: [] for m in self._AUTO_ORDER}})
        per = self._AUTO_TRIALS + 1
        mode = self._AUTO_ORDER[st["i"] // per]
        t0 = time.perf_counter()
        h = self.step_host(host_actions, mode=mode, packed=packed)
        if st["i"] % per:                       # the first call of each mode allocates / warms up: not timed
            st["t"][mode].append(time.perf_counter() - t0)
        st["i"] += 1
        if st["i"] == per * len(self._AUTO_ORDER):
            self.__dict__.setdefault("_auto_choices", {})[packed] = min(
                self._AUTO_ORDER, key=lambda m: sorted(st["t"][m])[len(st["t"][m]) // 2])
            self.auto_mode_times = {m: sorted(v)[len(v) // 2] for m, v in st["t"].items()}
        return h

    def synchronize(self) -> None:
        """Wait for the launches enqueued so far (needed before reading ``pinned_outputs`` tensors on the host)."""
        torch.cuda.current_stream(self.device).synchronize()

    def observe(self) -> None:
        _lib.check(self.L.cat_env_observe(self._h, self.state.data_ptr(), C.byref(self._io), self._stream()),
                   "cat_env_observe")

    # ------------------------------------------------------------------ frames (render.py)
    def positions(self) -> torch.Tensor:
        """(N, A, 2) float32 view of the agents' positions inside the packed state buffer (words 0 .. 2A-1 of each
        world's record): read-only use, no copy."""
        return self.state.view(torch.float32).as_strided((self.n_worlds, self.A, 2), (self.info.record_words, 2, 1))

    def renderer(self):
        """The ``render.Renderer`` of this environment's maps, created on first use (outside graph capture)."""
        if getattr(self, "_renderer", None) is None:
            from .render import Renderer
            self._renderer = Renderer(self.cmaps, self.R, self.device)
        return self._renderer

    def render_frames(self, worlds=None, rays: bool = False, downsample: int = 1, out: Optional[torch.Tensor] = None,
                      agent_radius: float = 5.0) -> torch.Tensor:
        """``rgb_array`` frames (K, W', H', 3) uint8 on the device of the worlds ``worlds`` (None: every world; a
        sequence or an int64 tensor, on the device under graph capture), one launch on the current stream; each frame is
        ``render.render_rgb`` of the world's own map, zero-padded to the largest window, downsampled as
        ``frame[d//2::d, d//2::d]``.

        ``rays=True`` draws each agent's sensor rays as its sensor reports them from the drawn positions: it first runs
        ``cat_env_observe`` into a private record buffer (observing writes no state back), so the environment's own
        outputs are untouched, and for a world that does not end in the next step the overlay is that step's
        observation bit for bit.  The renderer and the private buffer are created by the first call, which must
        therefore happen outside CUDA-graph capture (as ``step_host``'s buffers do); later calls allocate nothing when
        ``out`` is given and ``worlds`` is None or a device tensor."""
        if worlds is not None and not (isinstance(worlds, torch.Tensor) and worlds.device == self.device
                                       and worlds.dtype == torch.int64):
            worlds = torch.as_tensor(worlds, dtype=torch.int64).reshape(-1).to(self.device)
        return self.renderer().render(self.positions(), world=worlds, map_of=self.map_index,
                                      rays=self.sensor_rays() if rays else None, downsample=downsample,
                                      agent_radius=agent_radius, out=out)

    def sensor_rays(self):
        """(obs_dist (N, A, R) float16, obs_type (N, A, R) uint8): what every agent's sensor reports from the current
        positions, written by ``cat_env_observe`` into a private record buffer (created by the first call) on the
        current stream.  Neither the state nor the environment's outputs change.  The step computes its observation
        before it moves the agents, so for a world that does not end in the next step this is that step's observation."""
        if getattr(self, "_sensor_rec", None) is None:
            self._sensor_rec = torch.zeros(self.n_worlds * self.record_bytes, dtype=torch.uint8, device=self.device)
            self._sensor_io = CatStepIO(record=self._sensor_rec.data_ptr(), record_world_stride=self.record_bytes)
            v = self._record_views(self._sensor_rec)
            self._sensor_views = (v["obs_dist"], v["obs_type"])
        _lib.check(self.L.cat_env_observe(self._h, self.state.data_ptr(), C.byref(self._sensor_io), self._stream()),
                   "cat_env_observe")
        return self._sensor_views

    # ------------------------------------------------------------------ state access (parity tests, checkpoints)
    def _view_tensors(self) -> Dict[str, torch.Tensor]:
        N, A, P, dev, K = self.n_worlds, self.A, self.P, self.device, CAT_WALL_SLOTS
        return dict(
            pos=torch.zeros((N, A, 2), dtype=torch.float32, device=dev),
            vel=torch.zeros((N, A, 2), dtype=torch.float32, device=dev),
            vbias=torch.zeros((N, A, 2), dtype=torch.float32, device=dev),
            tc=torch.zeros((N, A, 2), dtype=torch.float32, device=dev),
            step_count=torch.zeros(N, dtype=torch.int32, device=dev),
            episode=torch.zeros(N, dtype=torch.int32, device=dev),
            wall_hull=torch.full((N, A, K), -1, dtype=torch.int32, device=dev),
            wall_age=torch.full((N, A, K), -1, dtype=torch.int32, device=dev),
            wall_jn=torch.zeros((N, A, K), dtype=torch.float32, device=dev),
            pair_age=torch.full((N, max(P, 1)), -1, dtype=torch.int32, device=dev),
            pair_jn=torch.zeros((N, max(P, 1)), dtype=torch.float32, device=dev),
        )

    def get_state(self) -> Dict[str, torch.Tensor]:
        t = self._view_tensors()
        view = CatStateView(*[t[name].data_ptr() for name, _ in CatStateView._fields_])
        _lib.check(self.L.cat_env_get_state(self._h, self.state.data_ptr(), C.byref(view), self._stream()),
                   "cat_env_get_state")
        return t

    def set_state(self, **fields: torch.Tensor) -> None:
        """Overwrite selected state fields (``pos``, ``vel``, ``vbias``, ``tc``, ``step_count``, ``episode``,
        ``wall_hull``+``wall_age``+``wall_jn``, ``pair_age``+``pair_jn``)."""
        proto = self._view_tensors()
        ptrs, keep = [], []
        for name, _ in CatStateView._fields_:
            if name in fields:
                t = torch.as_tensor(fields[name]).to(device=self.device, dtype=proto[name].dtype).contiguous()
                if t.numel() != proto[name].numel():
                    raise ValueError(f"{name}: expected {tuple(proto[name].shape)}, got {tuple(t.shape)}")
                keep.append(t)
                ptrs.append(t.data_ptr())
            else:
                ptrs.append(None)
        unknown = set(fields) - {n for n, _ in CatStateView._fields_}
        if unknown:
            raise ValueError(f"unknown state fields {sorted(unknown)}")
        view = CatStateView(*ptrs)
        _lib.check(self.L.cat_env_set_state(self._h, self.state.data_ptr(), C.byref(view), self._stream()),
                   "cat_env_set_state")
        torch.cuda.current_stream(self.device).synchronize()  # `keep` tensors must outlive the copy

    def episode_totals_raw(self, reset: bool = False) -> np.ndarray:
        """The per-map-slot ``CatEpisodeTotals`` as a numpy structured array (``episodes.TOTALS_DTYPE``), one copy to the
        host (which waits for the launches enqueued so far).  ``reset`` zeroes them on the device afterwards."""
        if self._episode_totals is None:
            raise _lib.CatError("episode statistics are off (want_episode_stats=False)")
        raw = np.frombuffer(self._episode_totals.cpu().numpy().tobytes(), dtype=episodes.TOTALS_DTYPE)
        if reset:
            self._episode_totals.zero_()
        return raw.copy()

    def episode_totals(self, reset: bool = False, agents: Optional[Sequence[str]] = None) -> list:
        """Every map slot's totals decoded (``episodes.summarize``: episodes, captures, timeouts, length and per-agent
        return moments); ``agents`` names the agents in index order (default ``0 .. A-1``)."""
        raw = self.episode_totals_raw(reset)
        agents = list(agents) if agents is not None else [str(i) for i in range(self.A)]
        return [episodes.summarize(raw[m], agents) for m in range(len(raw))]

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """Checkpoint = the packed state buffer (everything else is recomputed by ``observe``), and the running returns
        when episode statistics are on."""
        sd = {"state": self.state.clone(), "seed": torch.tensor(self.params["seed"])}
        if self.episode_acc is not None:
            sd["episode_acc"] = self.episode_acc.clone()
        if self._wp is not None:
            sd["world_params"] = self._wp.clone()
            sd["param_ranges"] = self._wp_ranges.clone()
        if self._script_mode is not None:
            sd["script_mode"] = self._script_mode.clone()
        return sd

    def load_state_dict(self, sd: Mapping[str, torch.Tensor]) -> None:
        self.state.copy_(sd["state"].to(self.device))
        self.set_seed(int(sd["seed"]))
        if self.episode_acc is not None and "episode_acc" in sd:
            self.episode_acc.copy_(sd["episode_acc"].to(self.device))
        if self._wp is not None and "world_params" in sd:
            self._wp.copy_(sd["world_params"].to(self.device))
            self._ranges_host = sd["param_ranges"].cpu().numpy().copy().view(wparams.RANGES_DTYPE).reshape(-1)
            self._upload_ranges()
        if self._script_mode is not None and "script_mode" in sd:
            self.set_script_table(sd["script_mode"])

    # ------------------------------------------------------------------ per-world parameters
    def world_params(self) -> Dict[str, torch.Tensor]:
        """Named device views of the per-world parameter table (writes through them reach the kernel):
        ``unit_velocity`` (N, 2) and ``max_speed`` (N, 2) float32 by team (``[:, 0]`` cops, ``[:, 1]`` thieves),
        ``termination_radius`` (N,) float32 and ``max_step_count`` (N,) int32.  The kernel does not check what it
        reads: ``set_world_params`` does."""
        if self._wp is None:
            raise _lib.CatError("per-world parameters are off (want_world_params=False)")
        f = self._wp.view(torch.float32)
        return dict(unit_velocity=f[:, 0:2], max_speed=f[:, 2:4], termination_radius=f[:, 4], max_step_count=self._wp[:, 5])

    def set_world_params(self, mask: Optional[torch.Tensor] = None, **values) -> None:
        """Write per-world parameters in place (a captured graph stays valid), for the worlds of the (N,) bool ``mask``
        (all if None): ``field=value`` with a number or a tensor broadcastable to the selected worlds; ``unit_velocity``
        and ``max_speed`` take one value for both teams or ``{"cop": .., "thief": ..}``.  Every value is checked
        (``world_params.check_values``) before anything is written.  The new values apply from each world's next step;
        a later re-spawn of a world whose map slot draws replaces them."""
        views = self.world_params()
        sel = slice(None) if mask is None else torch.as_tensor(mask, device=self.device).reshape(-1).bool()
        if mask is not None and sel.numel() != self.n_worlds:
            raise ValueError(f"mask needs {self.n_worlds} entries, got {sel.numel()}")
        writes = []
        for field, value in values.items():
            for col, v in wparams.per_team(field, value):
                wparams.check_values(field, v)
                dst = views[field] if col is None else views[field][:, col]
                writes.append((dst, torch.as_tensor(v, device=self.device).to(dst.dtype)))
        for dst, t in writes:
            dst[sel] = t

    def set_param_ranges(self, slot: Optional[int] = None, draw: bool = True,
                         **ranges: Union[float, Tuple[float, float], Mapping]) -> None:
        """Set the randomisation of map slot ``slot`` (every slot if None): ``field=(lo, hi)`` or ``field=value`` (pinned),
        per team for ``unit_velocity`` / ``max_speed`` (``max_speed={"thief": (125, 175)}``); fields and teams not named
        are pinned to the environment's values.  With ``draw``, every later re-spawn of a world of the slot draws its
        table entry from these ranges; ``draw=False`` leaves the table to the caller.  Written in place."""
        if self._wp is None:
            raise _lib.CatError("per-world parameters are off (want_world_params=False)")
        entry = wparams.ranges_entry(ranges, self.params, draw)
        slots = range(len(self.cmaps)) if slot is None else [int(slot)]
        for s in slots:
            if not 0 <= s < len(self.cmaps):
                raise IndexError(f"map slot {s} out of range (0..{len(self.cmaps) - 1})")
        for s in slots:
            self._ranges_host[s] = entry
        self._upload_ranges()

    def param_ranges(self) -> np.ndarray:
        """A copy of every map slot's ranges (``world_params.RANGES_DTYPE``)."""
        return self._ranges_host.copy()

    def _upload_ranges(self) -> None:
        words = torch.from_numpy(self._ranges_host.view(np.int32).reshape(len(self.cmaps), wparams.RANGE_WORDS).copy())
        self._wp_ranges.copy_(words)

    # ------------------------------------------------------------------ scripted agents
    def _require_scripts(self) -> None:
        if self._script_mode is None:
            raise _lib.CatError("scripted agents are off (want_scripts=False)")

    @property
    def script_modes(self) -> torch.Tensor:
        """(N, A) uint8 device table of every agent's mode, read by each step (``scripts.MODES``).  Write it with
        ``set_scripts``, which checks the values and keeps the host mirror that ``scripted_in`` answers from."""
        self._require_scripts()
        return self._script_mode

    @property
    def script_decisions(self) -> torch.Tensor:
        """(N, A) uint8 device table: what the random, chase and evade controllers decided (bits 0-1, 2-3, 4-5) from
        the observation the last step or reset emitted.  Written by the kernel."""
        self._require_scripts()
        return self._script_dec

    def scripted_actions(self) -> torch.Tensor:
        """(N, A) int64 next actions of the scripted agents (``scripts.decode``; -1 where an agent is not scripted)."""
        self._require_scripts()
        return cscripts.decode(self._script_dec, self._script_mode)

    def set_scripts(self, modes: Mapping[int, Union[str, int]], mask=None) -> None:
        """Set the mode of agents ``{agent index: mode}`` (a name of ``scripts.MODES`` or its code) in the worlds of the
        (N,) bool ``mask`` (all if None).  Everything is checked before anything is written; the table is written in
        place, so a captured graph stays valid, and the next step acts on the new modes."""
        self._require_scripts()
        codes = {}
        for a, mode in modes.items():
            if isinstance(a, bool) or not isinstance(a, (int, np.integer)) or not 0 <= int(a) < self.A:
                raise ValueError(f"agent index must be in 0..{self.A - 1}, got {a!r}")
            codes[int(a)] = cscripts.mode_code(mode)
        sel = None if mask is None else cscripts.check_mask(mask, self.n_worlds)
        for a, code in codes.items():
            if sel is None:
                self._script_mode[:, a] = code
                self._script_mode_host[:, a] = code
            else:
                self._script_mode[:, a].masked_fill_(sel.to(self.device), code)
                self._script_mode_host[sel.numpy(), a] = code

    def set_script_table(self, modes: torch.Tensor) -> None:
        """Replace the whole (N, A) mode table (codes 0..3, checked), in place, e.g. to restore a saved copy."""
        self._require_scripts()
        modes = torch.as_tensor(modes)
        cscripts.check_modes(modes)
        if tuple(modes.shape) != (self.n_worlds, self.A):
            raise ValueError(f"script modes must be ({self.n_worlds}, {self.A}), got {tuple(modes.shape)}")
        host = modes.to(torch.uint8).cpu()
        self._script_mode.copy_(host.to(self.device))
        self._script_mode_host[:] = host.numpy()

    def scripted_in(self, agent: int) -> str:
        """``"all"``, ``"none"`` or ``"some"``: in which worlds agent ``agent`` is scripted, from the host mirror of the
        modes (no device sync).  ``"none"`` without scripts."""
        if self._script_mode_host is None:
            return "none"
        col = self._script_mode_host[:, int(agent)] != 0
        return "all" if col.all() else "some" if col.any() else "none"
