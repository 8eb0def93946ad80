"""``rgb_array`` frames (replacement for ``base_env.py:481-510``; SURVEY.md f-4).

Visual only — never on the hot path.  A frame is shaped like ``pygame.surfarray.array3d(window)``: ``(width, height,
3)`` uint8, walls white on black (``pyproject.toml:21-23``), cops blue, thieves red (``cop.py:30``, ``thief.py:30``),
and optionally every agent's sensor rays under the walls, coloured by what each ray reports.

* ``render_rgb`` draws one world in numpy on the host.  It defines what a frame contains and is the reference the
  device renderer is tested against; it needs no GPU, so a saved trajectory can be redrawn anywhere.
* ``Renderer`` draws many worlds in one CUDA launch (``cat_render``), bit for bit the frames ``render_rgb`` draws.
* ``TrajectoryRecorder`` keeps chosen worlds' steps on the device and renders or saves them afterwards.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple, Union

import numpy as np

#: ray colour by ObjectType (WALL 0, COP 1, THIEF 2, EMPTY 4); rays of any other type are not drawn
RAY_COLORS = {0: (96, 96, 96), 1: (0, 160, 255), 2: (255, 160, 0), 4: (40, 40, 40)}


def _on_segment(cx, cy, px, py, qx, qy):
    """Pixel centres (cx, cy) within 0.5 of the segment P -> Q, in fp64 with every operation rounded (numpy never
    fuses): e = Q - P, w = C - P, t = w.e, L = e.e; t <= 0: |w|^2 <= 0.25; t >= L: |C - Q|^2 <= 0.25; else
    (w x e)^2 <= 0.25 L."""
    ex, ey = qx - px, qy - py
    wx, wy = cx - px, cy - py
    t = wx * ex + wy * ey
    L = ex * ex + ey * ey
    cr = wx * ey - wy * ex
    near_p = wx * wx + wy * wy <= 0.25
    near_q = (cx - qx) * (cx - qx) + (cy - qy) * (cy - qy) <= 0.25
    return np.where(t <= 0, near_p, np.where(t >= L, near_q, cr * cr <= 0.25 * L))


def _draw_rays(img: np.ndarray, pos: np.ndarray, dist, types, dirs) -> None:
    W, H = img.shape[:2]
    d = np.asarray(dist, np.float16).astype(np.float64)
    ty = np.asarray(types, np.uint8)
    u = np.asarray(dirs, np.float32).astype(np.float64)
    for a, (px, py) in enumerate(pos):
        for i in range(u.shape[0]):
            color = RAY_COLORS.get(int(ty[a, i]))
            if color is None:
                continue
            qx, qy = px + d[a, i] * u[i, 0], py + d[a, i] * u[i, 1]
            if not np.isfinite([px, py, qx, qy]).all():
                continue
            # every pixel whose centre can be within 0.5 of the segment, with a pixel to spare on each side
            x0, x1 = max(0, int(np.floor(min(px, qx))) - 2), min(W, int(np.floor(max(px, qx))) + 2)
            y0, y1 = max(0, int(np.floor(min(py, qy))) - 2), min(H, int(np.floor(max(py, qy))) + 2)
            if x1 <= x0 or y1 <= y0:
                continue
            xs, ys = np.meshgrid(np.arange(x0, x1) + 0.5, np.arange(y0, y1) + 0.5, indexing="ij")
            img[x0:x1, y0:y1][_on_segment(xs, ys, px, py, qx, qy)] = color


def render_rgb(cmap, pos: np.ndarray, agent_radius: float = 5.0, rays=None) -> np.ndarray:
    """One world as ``(width, height, 3)`` uint8.  ``rays=(dist, type, dirs)`` adds the sensor rays: ``dist`` (A, R)
    float16 and ``type`` (A, R) ObjectType as the observation holds them, ``dirs`` (R, 2) float32 ray directions
    (``ray_directions``).  Ray i of agent a is the segment from the agent's position P to P + dist[a, i] dirs[i]
    (fp64); a pixel is on it when its centre is within 0.5 of it, and where rays overlap the later (a, i) wins.
    Layers, each over the last: black, rays, walls, agents."""
    W, H = int(cmap.window[0]), int(cmap.window[1])
    img = np.zeros((W, H, 3), np.uint8)
    pos = np.asarray(pos, np.float64)
    if rays is not None:
        _draw_rays(img, pos, *rays)
    for h in range(cmap.n_hulls):
        o, e = cmap.hull_off[h], cmap.hull_off[h + 1]
        l, b, r, t = cmap.hull_bb[h]
        x0, x1 = max(0, int(np.floor(l - 1))), min(W, int(np.ceil(r + 1)) + 1)
        y0, y1 = max(0, int(np.floor(b - 1))), min(H, int(np.ceil(t + 1)) + 1)
        if x1 <= x0 or y1 <= y0:
            continue
        xs, ys = np.meshgrid(np.arange(x0, x1) + 0.5, np.arange(y0, y1) + 0.5, indexing="ij")
        inside = np.ones(xs.shape, bool)
        for (vx, vy), (nx, ny) in zip(cmap.vert[o:e], cmap.normal[o:e]):
            inside &= ((xs - vx) * nx + (ys - vy) * ny) <= 1.0  # wall radius 1
        img[x0:x1, y0:y1][inside] = (255, 255, 255)
    for a, (px, py) in enumerate(pos):
        color = (0, 0, 255) if a < cmap.n_cops else (255, 0, 0)
        x0, x1 = max(0, int(px - agent_radius - 1)), min(W, int(px + agent_radius + 2))
        y0, y1 = max(0, int(py - agent_radius - 1)), min(H, int(py + agent_radius + 2))
        if x1 <= x0 or y1 <= y0:
            continue
        xs, ys = np.meshgrid(np.arange(x0, x1) + 0.5, np.arange(y0, y1) + 0.5, indexing="ij")
        img[x0:x1, y0:y1][(xs - px) ** 2 + (ys - py) ** 2 <= agent_radius ** 2] = color
    return img


def ray_directions(n_rays: int) -> np.ndarray:
    """(R, 2) float32: the ray directions the step kernel and the renderer use (``cat_ray_directions``; host only)."""
    from . import _lib
    L = _lib.load()
    out = np.zeros((int(n_rays), 2), np.float32)
    _lib.check(L.cat_ray_directions(int(n_rays), _lib.np_ptr(out)), "cat_ray_directions")
    return out


def _byte_stride(t, dim: int) -> int:
    return t.stride(dim) * t.element_size()


class Renderer:
    """Device renderer over compiled maps (``cat_renderer_create``): frames of many worlds in one launch, equal bit
    for bit to ``render_rgb``.  Needs a CUDA device (no CPU fallback).  The frame is the size of the largest window of
    the maps; a frame of a smaller map is zero outside its window."""

    def __init__(self, cmaps, n_rays: int = 90, device="cuda:0"):
        import torch
        from . import _lib
        from .maps import CompiledMap
        from .worlds import _map_desc, _require_cuda
        self.cmaps = [cmaps] if isinstance(cmaps, CompiledMap) else list(cmaps)
        self.device = torch.device(device)
        _require_cuda(self.device)
        self.L = _lib.load()
        self.n_rays = int(n_rays)
        self.n_cops = self.cmaps[0].n_cops
        self.A = self.cmaps[0].n_cops + self.cmaps[0].n_thieves
        descs = [_map_desc(m) for m in self.cmaps]
        n = len(self.cmaps)
        mds = (_lib.CatMapDesc * n)(*[md for md, _ in descs])
        win = (C.c_int32 * (2 * n))(*[int(v) for m in self.cmaps for v in (m.window[0], m.window[1])])
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        h = C.c_void_p()
        _lib.check(self.L.cat_renderer_create(mds, win, n, self.n_rays, dev_index, C.byref(h)), "cat_renderer_create")
        self._h = h

    def frame_size(self, downsample: int = 1) -> Tuple[int, int]:
        from . import _lib
        w, h = C.c_int32(), C.c_int32()
        _lib.check(self.L.cat_renderer_frame_size(self._h, int(downsample), C.byref(w), C.byref(h)),
                   "cat_renderer_frame_size")
        return w.value, h.value

    def render(self, pos, world=None, map_of=None, rays=None, downsample: int = 1, agent_radius: float = 5.0,
               out=None):
        """Frames (K, W', H', 3) uint8 on the device, enqueued on the current stream.

        ``pos`` (E, A, 2) float32 on the device, agents at 8-byte steps (strides (s, 2, 1): a view of the packed state
        buffer works); ``world`` (K,) int64 on the device, the element of each frame (None: K = E, frame k shows
        element k; an id outside [0, E) gives a zero frame); ``map_of`` (E,) int64 on the device, each element's map
        (None: map 0); ``rays`` None or (dist (E, A, R) float16, type (E, A, R) uint8), both with strides (s, R, 1);
        ``out`` a contiguous (K, W', H', 3) uint8 tensor on the device to draw into (needed under graph capture)."""
        import torch
        from . import _lib
        E, A, R = pos.shape[0], self.A, self.n_rays

        def need(t, name, dtype, shape, inner):
            if t.dtype != dtype or t.device != self.device or tuple(t.shape) != shape or t.stride()[1:] != inner:
                raise ValueError(f"{name}: need {dtype} {shape} with inner strides {inner} on {self.device}, got "
                                 f"{t.dtype} {tuple(t.shape)} strides {t.stride()} on {t.device}")
        need(pos, "pos", torch.float32, (E, A, 2), (2, 1))
        io = _lib.CatRenderIO()
        io.n_elements, io.pos, io.pos_stride = E, pos.data_ptr(), _byte_stride(pos, 0)
        K = E
        if world is not None:
            need(world, "world", torch.int64, (world.shape[0],), ())
            if not world.is_contiguous():
                raise ValueError("world must be contiguous")
            K, io.world = world.shape[0], world.data_ptr()
        if map_of is not None:
            need(map_of, "map_of", torch.int64, (E,), ())
            if not map_of.is_contiguous():
                raise ValueError("map_of must be contiguous")
            io.map_of = map_of.data_ptr()
        if rays is not None:
            dist, types = rays
            need(dist, "ray dist", torch.float16, (E, A, R), (R, 1))
            need(types, "ray type", torch.uint8, (E, A, R), (R, 1))
            io.ray_dist, io.ray_dist_stride = dist.data_ptr(), _byte_stride(dist, 0)
            io.ray_type, io.ray_type_stride = types.data_ptr(), _byte_stride(types, 0)
        W, H = self.frame_size(downsample)
        if out is None:
            out = torch.empty((K, W, H, 3), dtype=torch.uint8, device=self.device)
        elif out.dtype != torch.uint8 or out.device != self.device or tuple(out.shape) != (K, W, H, 3) or not out.is_contiguous():
            raise ValueError(f"out: need a contiguous uint8 ({K}, {W}, {H}, 3) tensor on {self.device}")
        io.n_frames, io.downsample, io.agent_radius, io.frames = K, int(downsample), float(agent_radius), out.data_ptr()
        if K:
            _lib.check(self.L.cat_render(self._h, C.byref(io), torch.cuda.current_stream(self.device).cuda_stream),
                       "cat_render")
        return out

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.L.cat_renderer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TrajectoryRecorder:
    """Records chosen worlds of an environment (``BatchedCopsThievesEnv`` or ``CatWorlds``) step by step, on the device.

    Call ``record()`` after each step: it enqueues device work only (``index_select`` into slot t, no host sync): the
    worlds' positions and maps, with ``rays`` what their sensors report from those positions (``CatWorlds.sensor_rays``,
    one extra observe launch: the observation a step returns was taken before it moved the agents), and the step's
    rewards, terminated, truncated and winner.  ``frames()`` renders recorded steps in one launch; ``save()`` writes an ``.npz`` that ``render_rgb``
    can redraw without a GPU (``redraw``).  Both raise if the environment replaced a map (``set_map``) after recording
    began: the recorded map indices would then name the new map."""

    def __init__(self, env, worlds: Union[Sequence[int], "object"], capacity: int, rays: bool = True):
        import torch
        self.w = env.worlds if hasattr(env, "worlds") else env
        w = self.w
        self.worlds = torch.as_tensor(worlds, dtype=torch.int64).reshape(-1).to(w.device)
        self.capacity, self.rays, self.t = int(capacity), bool(rays), 0
        T, K, A, R, dev = self.capacity, self.worlds.numel(), w.A, w.R, w.device
        self.pos = torch.zeros((T, K, A, 2), dtype=torch.float32, device=dev)
        self.map_of = torch.zeros((T, K), dtype=torch.int64, device=dev)
        self.obs_dist = torch.zeros((T, K, A, R), dtype=torch.float16, device=dev) if rays else None
        self.obs_type = torch.zeros((T, K, A, R), dtype=torch.uint8, device=dev) if rays else None
        self.reward = torch.zeros((T, K, A), dtype=torch.float32, device=dev)
        self.terminated = torch.zeros((T, K), dtype=torch.uint8, device=dev)
        self.truncated = torch.zeros((T, K), dtype=torch.uint8, device=dev)
        self.winner = torch.zeros((T, K), dtype=torch.int8, device=dev)

    def record(self) -> None:
        import torch
        if self.t >= self.capacity:
            raise IndexError(f"the recorder is full ({self.capacity} steps)")
        w, t, idx = self.w, self.t, self.worlds
        if t == 0:
            self._maps_replaced = w.maps_replaced
        torch.index_select(w.positions(), 0, idx, out=self.pos[t])
        torch.index_select(w.map_index, 0, idx, out=self.map_of[t])
        if self.rays:
            dist, types = w.sensor_rays()
            torch.index_select(dist, 0, idx, out=self.obs_dist[t])
            torch.index_select(types, 0, idx, out=self.obs_type[t])
        torch.index_select(w.reward, 0, idx, out=self.reward[t])
        torch.index_select(w.terminated, 0, idx, out=self.terminated[t])
        torch.index_select(w.truncated, 0, idx, out=self.truncated[t])
        torch.index_select(w.winner, 0, idx, out=self.winner[t])
        self.t += 1

    def _check_maps(self) -> None:
        if self.t and self.w.maps_replaced != self._maps_replaced:
            raise RuntimeError("the environment replaced a map (set_map) after this recording began: its map indices "
                               "no longer name the maps the steps ran on")

    def frames(self, start: int = 0, stop: Optional[int] = None, downsample: int = 1):
        """(stop - start, K, W', H', 3) uint8 frames of the recorded steps [start, stop), one launch."""
        self._check_maps()
        stop = self.t if stop is None else min(int(stop), self.t)
        n, K, A, R = max(0, stop - start), self.worlds.numel(), self.w.A, self.w.R
        rays = None
        if self.rays:
            rays = (self.obs_dist[start:stop].reshape(n * K, A, R), self.obs_type[start:stop].reshape(n * K, A, R))
        out = self.w.renderer().render(self.pos[start:stop].reshape(n * K, A, 2),
                                       map_of=self.map_of[start:stop].reshape(n * K), rays=rays, downsample=downsample)
        return out.reshape(n, K, *out.shape[1:])

    def save(self, path) -> None:
        """``.npz`` of the recorded steps, with the map names and ray directions ``redraw`` needs."""
        self._check_maps()
        t = self.t
        arrays = dict(worlds=self.worlds.cpu().numpy(), map_names=np.array([c.name for c in self.w.cmaps]),
                      windows=np.array([c.window for c in self.w.cmaps], np.int32),
                      ray_dirs=ray_directions(self.w.R), pos=self.pos[:t].cpu().numpy(),
                      map_of=self.map_of[:t].cpu().numpy(), reward=self.reward[:t].cpu().numpy(),
                      terminated=self.terminated[:t].cpu().numpy(), truncated=self.truncated[:t].cpu().numpy(),
                      winner=self.winner[:t].cpu().numpy())
        if self.rays:
            arrays.update(obs_dist=self.obs_dist[:t].cpu().numpy(), obs_type=self.obs_type[:t].cpu().numpy())
        np.savez_compressed(path, **arrays)


def redraw(rec, t: int, k: int, agent_radius: float = 5.0, cmaps=None) -> np.ndarray:
    """Frame of step ``t``, world ``k`` of a saved recording (``np.load`` of ``TrajectoryRecorder.save``) through
    ``render_rgb`` on the host: the world's own map, its own window.  ``cmaps``: the compiled maps, default the built-in
    maps of ``rec["map_names"]``."""
    if cmaps is None:
        from .maps import compile_map, load_named_map
        cmaps = [compile_map(load_named_map(str(n))) for n in rec["map_names"]]
    rays = None
    if "obs_dist" in rec:
        rays = (rec["obs_dist"][t, k], rec["obs_type"][t, k], rec["ray_dirs"])
    return render_rgb(cmaps[int(rec["map_of"][t, k])], rec["pos"][t, k], agent_radius, rays=rays)
