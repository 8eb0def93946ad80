"""Map loader and map compiler (host side, init-time only).

Mirrors the reference ``Map`` (``/root/reference/src/maps/map.py:10-128``): same constructor,
same public attributes (``window_dimensions``, ``canvas_dimensions``, ``cops_count``,
``thieves_count``, ``cops_positions``, ``thieves_positions``, ``agent_spawn_regions``), same
block rules (rect -> 5-vertex closed ring with ``w``/``h`` defaulting to 1 and negative extents
allowed, ``map.py:37-52``; poly -> the listed vertices, ``map.py:53-58``).

What the reference does with the blocks afterwards lives in third-party code:
``pymunk.Poly(space.static_body, vs, radius=1)`` (``map.py:125-128``) runs Chipmunk2D's
``cpConvexHull(tol=0)`` over the ring, so every block becomes the *convex hull* of its vertices,
CCW, collinear points dropped, inflated by radius 1.  ``compile_map`` restates that and lays the
result out as flat arrays for the CUDA kernels (and, in fp64, for the CPU oracle).

No shapely / pymunk / pygame dependency.
"""
from __future__ import annotations

import json
import math
from dataclasses import dataclass, field
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

MAPS_DATA_DIR = Path(__file__).resolve().parent / "maps_data"

#: hull radius every wall polygon gets in the reference (``map.py:127``)
WALL_RADIUS = 1.0


def builtin_map_path(name: str) -> Path:
    """Path of a map shipped with the package (normalised ``catmap-1`` schema)."""
    p = MAPS_DATA_DIR / f"{name}.catmap.json"
    if not p.exists():
        raise FileNotFoundError(f"no built-in map {name!r} under {MAPS_DATA_DIR}")
    return p


def _rect_ring(blk: dict) -> List[Tuple[float, float]]:
    # map.py:37-52 — x,y required; w,h optional (default 1); closed 5-vertex ring
    x, y = blk.get("x"), blk.get("y")
    if x is None or y is None:
        raise ValueError("x and y coordinates are required for rectangle blocks.")
    w = blk.get("w") if blk.get("w") is not None else 1
    h = blk.get("h") if blk.get("h") is not None else 1
    return [(x, y), (x + w, y), (x + w, y + h), (x, y + h), (x, y)]


def _parse_block(blk: dict) -> List[Tuple[float, float]]:
    blk_type = blk.get("type", "rect")  # map.py:36 — default to rect
    if blk_type == "rect":
        return _rect_ring(blk)
    if blk_type == "poly":
        vs = blk.get("vs")
        if vs is None:
            raise ValueError("Vertices are required for polygon blocks.")
        return [(v.get("x"), v.get("y")) for v in vs]
    raise ValueError(f"Unknown block type: {blk_type}")


class Map:
    """Drop-in for the reference ``maps.Map`` (``map.py:10``).

    ``Map(path)`` accepts the reference's ``maps_templates`` JSON schema and this package's
    normalised ``catmap-1`` schema (what ``tools/import_maps.py`` writes).  Two extensions that the
    reference does not have, both keyword-only and off by default:

    * ``scale=(sx, sy)`` multiplies every block/agent/region coordinate (needed for
      ``labyrinth.json`` whose blocks are in 30x20 canvas cells, SURVEY.md §7 hard part 8);
    * ``agents=[{"type": "cop", "x":..., "y":..., "spawn_regions": [...]}, ...]`` injects or
      replaces the agent list (``labyrinth.json`` has no ``agents`` key and the reference raises
      ``KeyError`` on it, ``map.py:75`` — so does this class unless ``agents`` is given).
    """

    def __init__(self, map_path, *, scale: Optional[Tuple[float, float]] = None,
                 agents: Optional[Sequence[dict]] = None) -> None:
        self.map_path = str(map_path)
        self.unit_size = 5.0
        self.blocks: List[List[Tuple[float, float]]] = []
        self.agent_spawn_regions: Dict[str, List[dict]] = {}
        with open(self.map_path, "r") as f:
            self._parse_map_data(json.load(f), scale, agents)

    @classmethod
    def from_dict(cls, data: dict, name: str) -> "Map":
        """A map from an already parsed JSON document of either schema ``Map(path)`` reads (``catmap-1`` or the
        reference's); ``name`` stands in for the file name (``compile_map`` names the compiled map after it)."""
        m = cls.__new__(cls)
        m.map_path = str(name)
        m.unit_size = 5.0
        m.blocks, m.agent_spawn_regions = [], {}
        m._parse_map_data(data, None, None)
        return m

    def to_dict(self) -> dict:
        """The ``catmap-1`` document of this map (what ``Map.from_dict`` and ``Map(path)`` read back)."""
        counts: Dict[str, int] = {}
        agents = []
        for a in self._agents:
            idx = counts.get(a["type"], 0)
            counts[a["type"]] = idx + 1
            regs = self.agent_spawn_regions.get(f"{a['type']}_{idx}")
            agents.append({"type": a["type"], "pos": [a["x"], a["y"]],
                           **({"regions": [[r["x"], r["y"], r["w"], r["h"]] for r in regs]} if regs else {})})
        return {"format": "catmap-1", "window": list(self.window_dimensions), "canvas": list(self.canvas_dimensions),
                "blocks": [[c for v in ring for c in v] for ring in self.blocks], "agents": agents}

    # ------------------------------------------------------------------ parsing
    def _parse_map_data(self, data: dict, scale, agents_override) -> None:
        if data.get("format") == "catmap-1":
            self.window_dimensions = tuple(data["window"])
            self.canvas_dimensions = tuple(data["canvas"])
            rings = [list(zip(b[0::2], b[1::2])) for b in data["blocks"]]
            agents = data.get("agents")
            if agents is not None:
                agents = [
                    {"type": a["type"], "x": a["pos"][0], "y": a["pos"][1],
                     **({"spawn_regions": [dict(x=r[0], y=r[1], w=r[2], h=r[3]) for r in a["regions"]]}
                        if a.get("regions") else {})}
                    for a in agents
                ]
        else:
            self.window_dimensions = tuple(data["window"].values())  # map.py:71
            self.canvas_dimensions = tuple(data["canvas"].values())  # map.py:72
            rings = [_parse_block(b) for b in data["objects"]["blocks"]]
            agents = data.get("agents")
        if agents_override is not None:
            agents = [dict(a) for a in agents_override]
        if agents is None:
            raise KeyError("agents")  # map.py:75 behaviour

        sx, sy = (1.0, 1.0) if scale is None else (float(scale[0]), float(scale[1]))
        self.scale = (sx, sy)
        self.blocks = [[(vx * sx, vy * sy) for vx, vy in ring] for ring in rings]

        counts: Dict[str, int] = {}
        self.agent_spawn_regions = {}
        scaled_agents = []
        for agent in agents:
            a = dict(agent)
            if scale is not None and agents_override is None:
                a["x"], a["y"] = a["x"] * sx, a["y"] * sy
            atype = a["type"]
            idx = counts.get(atype, 0)
            agent_id = f"{atype}_{idx}"
            regions = None
            if "spawn_regions" in a:  # map.py:82-97 (plural first)
                sd = a["spawn_regions"]
                if isinstance(sd, list) and all(isinstance(it, dict) for it in sd):
                    regions = sd
                elif isinstance(sd, dict):
                    regions = [sd]
            elif "spawn_region" in a:  # map.py:98-106
                sd = a["spawn_region"]
                if isinstance(sd, dict):
                    regions = [sd]
            if regions is not None:
                for r in regions:
                    assert all(k in r for k in ("x", "y", "w", "h")), \
                        "Invalid spawn region format. Must contain x, y, w, h."
                self.agent_spawn_regions[agent_id] = [dict(r) for r in regions]
            counts[atype] = idx + 1
            scaled_agents.append(a)
        self._agents = scaled_agents
        self.cops_positions = [(a["x"], a["y"]) for a in scaled_agents if a["type"] == "cop"]
        self.thieves_positions = [(a["x"], a["y"]) for a in scaled_agents if a["type"] == "thief"]
        self.cops_count = len(self.cops_positions)
        self.thieves_count = len(self.thieves_positions)

    def populate_space(self, space) -> None:  # map.py:119
        raise RuntimeError(
            "Map.populate_space() fills a pymunk.Space; the B200 build has no Pymunk space — "
            "walls are compiled with compile_map() and staged into GPU shared memory instead.")


# ---------------------------------------------------------------------------------- hulls
def convex_hull_ccw(points: Sequence[Tuple[float, float]]) -> np.ndarray:
    """Convex hull, counter-clockwise (cross > 0), duplicates and collinear points dropped.

    Restates what ``cpConvexHull(count, verts, result, NULL, tol=0.0)`` yields for
    ``pymunk.Poly`` (SURVEY.md A.9): the hull as a *set* is unique, and Chipmunk's QuickHull with
    ``tol=0`` keeps only strict extreme points.  Only the starting vertex may differ, which does
    not change any query result (plane indexing matters only for exact ties).
    """
    pts = sorted(set((float(x), float(y)) for x, y in points))
    if len(pts) < 3:
        raise ValueError(f"degenerate block with {len(pts)} distinct vertices")

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    lower: List[Tuple[float, float]] = []
    for p in pts:
        while len(lower) >= 2 and cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    upper: List[Tuple[float, float]] = []
    for p in reversed(pts):
        while len(upper) >= 2 and cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    hull = lower[:-1] + upper[:-1]
    if len(hull) < 3:
        raise ValueError("degenerate (collinear) block")
    return np.asarray(hull, dtype=np.float64)


@dataclass
class CompiledMap:
    """Flat, device-ready description of one map (all fp64 here; the C library narrows to fp32).

    Edge ``i`` of a hull runs ``v[i-1] -> v[i]`` with outward unit normal ``n[i] = rperp(v[i] -
    v[i-1])/len`` — the ``planes[i]`` convention of Chipmunk's ``cpPolyShape`` (SURVEY.md A.7).
    """
    name: str
    window: Tuple[float, float]
    n_cops: int
    n_thieves: int
    hull_off: np.ndarray          # int32 [H+1] offsets into the edge arrays
    vert: np.ndarray              # f64 [E,2] hull vertices, CCW per hull
    normal: np.ndarray            # f64 [E,2] outward normal of edge ending at vert[i]
    edge_len: np.ndarray          # f64 [E]
    hull_bb: np.ndarray           # f64 [H,4] (l,b,r,t) of the raw hull vertices (un-inflated)
    init_pos: np.ndarray          # f64 [A,2] cops first, then thieves (base_env.py:91-96)
    region_off: np.ndarray        # int32 [A+1]
    regions: np.ndarray           # f64 [R,4] x,y,w,h
    # uniform grid over the hulls (+margin)
    grid_x0: float = 0.0
    grid_y0: float = 0.0
    cell: float = 32.0
    nx: int = 1
    ny: int = 1
    edge_hull: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))        # hull of each edge
    con_cell_off: np.ndarray = field(default_factory=lambda: np.zeros(2, np.int32))
    con_cell_hulls: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    # per grid cell: the edges a sensor sweep from ANY point of the cell can have as candidates (facing the
    # point and within view_range of it), nearest first — a conservative superset, the kernel still runs the
    # exact per-origin test on each listed edge
    view_cell_off: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    view_cell_edges: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    view_range: float = 0.0

    @property
    def n_hulls(self) -> int:
        return len(self.hull_off) - 1

    @property
    def n_edges(self) -> int:
        return int(self.hull_off[-1])

    @property
    def n_agents(self) -> int:
        return self.n_cops + self.n_thieves

    @property
    def agent_ids(self) -> List[str]:
        return [f"cop_{i}" for i in range(self.n_cops)] + [f"thief_{i}" for i in range(self.n_thieves)]


def _cells_touching_hull(verts, normals, bb, rho, gx0, gy0, cell, nx, ny) -> np.ndarray:
    """Conservative set of grid cells that may contain a point within ``rho`` of the hull.

    A cell is kept iff it overlaps the hull AABB grown by rho and is not entirely beyond any one
    of the hull's planes offset by rho.  Both tests only ever over-include, so every cell that
    really touches ``hull (+) rho`` is listed.
    """
    ix0 = max(0, int(math.floor((bb[0] - rho - gx0) / cell)))
    ix1 = min(nx - 1, int(math.floor((bb[2] + rho - gx0) / cell)))
    iy0 = max(0, int(math.floor((bb[1] - rho - gy0) / cell)))
    iy1 = min(ny - 1, int(math.floor((bb[3] + rho - gy0) / cell)))
    if ix1 < ix0 or iy1 < iy0:
        return np.zeros(0, np.int64)
    ix, iy = np.meshgrid(np.arange(ix0, ix1 + 1), np.arange(iy0, iy1 + 1), indexing="xy")
    ix, iy = ix.ravel(), iy.ravel()
    cx0, cy0 = gx0 + ix * cell, gy0 + iy * cell
    keep = np.ones(ix.shape, bool)
    for (vx, vy), (nx_, ny_) in zip(verts, normals):
        # most-inside corner of the cell w.r.t. this plane
        px = np.where(nx_ >= 0, cx0, cx0 + cell)
        py = np.where(ny_ >= 0, cy0, cy0 + cell)
        keep &= ((px - vx) * nx_ + (py - vy) * ny_) <= rho
    return (iy[keep] * nx + ix[keep]).astype(np.int64)


def _morton_sorted(hulls: List[np.ndarray]) -> List[np.ndarray]:
    """Order hulls along a Z-curve of their centroids (stable for ties).  Hull ids are internal to the
    compiled map (oracle and CUDA receive the same one), so any fixed order is as good as the file's."""
    c = np.asarray([h.mean(axis=0) for h in hulls])
    lo, span = c.min(axis=0), np.maximum(c.max(axis=0) - c.min(axis=0), 1e-9)
    q = np.minimum(((c - lo) / span * 65535.0).astype(np.int64), 65535)

    def spread(v):
        out = 0
        for b in range(16):
            out |= ((int(v) >> b) & 1) << (2 * b)
        return out
    keys = [spread(x) | (spread(y) << 1) for x, y in q]
    order = sorted(range(len(hulls)), key=lambda i: (keys[i], i))
    return [hulls[i] for i in order]


def choose_cell_size(hull_bb: np.ndarray, n_hulls: int) -> float:
    """Heuristic from the B200 sweeps (profiles/): ~4 cells per hull, clamped to [24, 200] units."""
    w = float(hull_bb[:, 2].max() - hull_bb[:, 0].min())
    h = float(hull_bb[:, 3].max() - hull_bb[:, 1].min())
    c = math.sqrt(max(w * h, 1.0) / (4.0 * max(n_hulls, 1)))
    return float(min(200.0, max(24.0, c)))


def view_lists(vert: np.ndarray, normal: np.ndarray, hull_off: np.ndarray, gx0: float, gy0: float, cell: float,
               nx: int, ny: int, view_range: float, eps: float = 1e-2) -> Tuple[np.ndarray, np.ndarray]:
    """Per grid cell, the edges that can be sensor candidates for SOME origin inside the cell.

    The kernel's per-origin candidate test is ``(pd > 0 or pdn > 0) and dist(origin, segment) < range`` with
    pd / pdn the signed distances to the edge's plane and to the next plane of the hull (they share the
    bevelled vertex).  Over a rectangular cell the first part is a union of two half-planes (a linear function
    is maximal at a corner) and the second is the distance between two convex sets (attained at a vertex of
    one of them), so both are evaluated exactly here, with ``eps`` of slack for the kernel's fp32.  Each list is
    ordered by distance from the cell centre, nearest first, so that near walls reach the depth buffer first.
    """
    E = len(vert)
    prev = np.zeros(E, np.int64)
    nxt = np.zeros(E, np.int64)
    for h in range(len(hull_off) - 1):
        o, e = int(hull_off[h]), int(hull_off[h + 1])
        idx = np.arange(o, e)
        prev[o:e] = np.roll(idx, 1)
        nxt[o:e] = np.roll(idx, -1)
    A, B, n, nn = vert[prev], vert, normal, normal[nxt]
    AB = B - A
    L2 = np.maximum((AB ** 2).sum(1), 1e-300)
    off = np.zeros(nx * ny + 1, np.int32)
    chunks = []
    for cy in range(ny):
        for cx in range(nx):
            # the cell rectangle, grown a little: the kernel bins the origin in fp32
            l, b = gx0 + cx * cell - 0.05, gy0 + cy * cell - 0.05
            r, t = l + cell + 0.1, b + cell + 0.1
            corners = np.array([[l, b], [r, b], [r, t], [l, t]])
            rel = corners[:, None, :] - B[None, :, :]
            facing = (np.einsum("ced,ed->ce", rel, n).max(0) > -eps) | (np.einsum("ced,ed->ce", rel, nn).max(0) > -eps)

            def to_rect(P):
                dx = np.maximum(np.maximum(l - P[:, 0], P[:, 0] - r), 0.0)
                dy = np.maximum(np.maximum(b - P[:, 1], P[:, 1] - t), 0.0)
                return np.hypot(dx, dy)
            d = np.minimum(to_rect(A), to_rect(B))
            for c in corners:
                tt = np.clip(((c - A) * AB).sum(1) / L2, 0.0, 1.0)
                q = A + AB * tt[:, None]
                d = np.minimum(d, np.hypot(c[0] - q[:, 0], c[1] - q[:, 1]))
            # a segment crossing the cell has distance 0: it then has an end point or a crossing inside, and the
            # corner-to-segment distances above are < the cell diagonal < any sensible range, so it is listed anyway
            sel = np.nonzero(facing & (d < view_range + eps))[0]
            ctr = np.array([(l + r) / 2, (b + t) / 2])
            tt = np.clip(((ctr - A[sel]) * AB[sel]).sum(1) / L2[sel], 0.0, 1.0)
            q = A[sel] + AB[sel] * tt[:, None]
            order = np.argsort(np.hypot(ctr[0] - q[:, 0], ctr[1] - q[:, 1]), kind="stable")
            chunks.append(sel[order].astype(np.int32))
            off[cy * nx + cx + 1] = off[cy * nx + cx] + len(sel)
    flat = np.concatenate(chunks) if chunks else np.zeros(0, np.int32)
    return off, flat


def _clip_interval(p0: np.ndarray, dp: np.ndarray, lo: np.ndarray, hi: np.ndarray):
    """Parameter interval of ``p0 + lam * dp`` (lam in R) inside the slab [lo, hi]; empty slabs give lo > hi."""
    with np.errstate(divide="ignore", invalid="ignore"):
        a, b = (lo - p0) / dp, (hi - p0) / dp
    l0, l1 = np.minimum(a, b), np.maximum(a, b)
    par = dp == 0.0
    inside = (p0 >= lo) & (p0 <= hi)
    l0 = np.where(par, np.where(inside, -np.inf, np.inf), l0)
    l1 = np.where(par, np.where(inside, np.inf, -np.inf), l1)
    return l0, l1


RAY_LIST_LB_SCALE = 64.0     # the lower bounds stored with the list entries are in 1/64 units, rounded down


def ray_lists(cmap: "CompiledMap", n_rays: int, ray_length: float, rsum: float, eps: float = 1e-2,
              grid: Optional[Tuple[float, float, float, int, int]] = None, return_bounds: bool = False):
    """Per (grid cell, ray index): the edges ray ``i`` cast from ANY origin inside the cell can touch, nearest first.

    The sensor's rays have fixed directions (``entity.py:182``), so for one direction the fat rays of every origin in
    a cell sweep the cell translated along that direction — in the ray's own frame (t along, w across) a region inside
    the rectangle ``[t0, t1 + L] x [w0, w1]`` of the cell's projections.  An edge (its plane offset by ``rsum`` and the
    bevel circle of radius ``rsum`` at its end vertex) can only be hit if its segment comes within ``rsum`` of that
    region, if the ray runs against its normal or the next edge's (the bevel's exposed arc spans the two), and if some
    point of the cell lies in front of one of those two planes.  Each entry carries a lower bound of the hit distance
    (quantised downwards): entries are sorted by it and the kernel stops walking a list as soon as the nearest hit it
    holds is closer than the next bound.  The list is a conservative superset and every listed edge still gets the
    exact ``cpPolyShapeSegmentQuery`` arithmetic, so results do not depend on it.

    This is the numpy statement of what the library builds in C++ at ``cat_env_create`` (``csrc/ray_lists.h``;
    ``tests/test_maps.py`` compares the two on the library's own grid, passed as ``grid = (x0, y0, cell, nx, ny)``;
    default: the compiled map's contact grid).

    Returns ``(off int32 [ncell * R + 1], ent uint32)`` with ``ent = (lb_q << 16) | edge`` (``lb_q`` in 1/64 units), plus
    the un-quantised bounds (float64, same order) when ``return_bounds``.
    """
    E, R, L = cmap.n_edges, int(n_rays), float(ray_length)
    assert E < 65536
    rs = rsum + eps
    vert, normal = cmap.vert, cmap.normal
    prev = np.zeros(E, np.int64)
    nxt = np.zeros(E, np.int64)
    for h in range(cmap.n_hulls):
        o, e = int(cmap.hull_off[h]), int(cmap.hull_off[h + 1])
        idx = np.arange(o, e)
        prev[o:e] = np.roll(idx, 1)
        nxt[o:e] = np.roll(idx, -1)
    A, B, n, nn = vert[prev], vert, normal, normal[nxt]
    gx0, gy0, cell, nx, ny = (cmap.grid_x0, cmap.grid_y0, cmap.cell, cmap.nx, cmap.ny) if grid is None else grid
    nx, ny = int(nx), int(ny)
    ncell = nx * ny
    cxs, cys = np.meshgrid(np.arange(nx), np.arange(ny), indexing="xy")
    cl = (gx0 + cxs.ravel() * cell - 0.05)[:, None]      # the kernel bins the origin in fp32: grow a little
    cb = (gy0 + cys.ravel() * cell - 0.05)[:, None]
    cr, ct = cl + cell + 0.1, cb + cell + 0.1
    corners = [(cl, cb), (cr, cb), (cr, ct), (cl, ct)]
    # ---- per (cell, edge), direction independent
    pd = np.full((ncell, E), -np.inf)
    pdn = np.full((ncell, E), -np.inf)
    for x, y in corners:
        pd = np.maximum(pd, (x - B[None, :, 0]) * n[None, :, 0] + (y - B[None, :, 1]) * n[None, :, 1])
        pdn = np.maximum(pdn, (x - B[None, :, 0]) * nn[None, :, 0] + (y - B[None, :, 1]) * nn[None, :, 1])
    in_front = (pd > -eps) | (pdn > -eps)
    # Euclidean distance cell rectangle <-> segment AB (0 if they intersect)
    AB = B - A
    L2 = np.maximum((AB ** 2).sum(1), 1e-300)

    def to_rect(P):
        dx = np.maximum(np.maximum(cl - P[None, :, 0], P[None, :, 0] - cr), 0.0)
        dy = np.maximum(np.maximum(cb - P[None, :, 1], P[None, :, 1] - ct), 0.0)
        return np.hypot(dx, dy)
    dist = np.minimum(to_rect(A), to_rect(B))
    for x, y in corners:
        tt = np.clip(((x - A[None, :, 0]) * AB[None, :, 0] + (y - A[None, :, 1]) * AB[None, :, 1]) / L2[None, :], 0.0, 1.0)
        dist = np.minimum(dist, np.hypot(x - (A[None, :, 0] + AB[None, :, 0] * tt), y - (A[None, :, 1] + AB[None, :, 1] * tt)))
    x0, x1 = _clip_interval(A[None, :, 0], AB[None, :, 0], cl, cr)
    y0, y1 = _clip_interval(A[None, :, 1], AB[None, :, 1], cb, ct)
    crosses = np.maximum(np.maximum(x0, y0), 0.0) <= np.minimum(np.minimum(x1, y1), 1.0)
    dist = np.where(crosses, 0.0, dist)
    lb_euclid = dist - rs

    cells_all, rays_all, lbs_all, edges_all, raw_all = [], [], [], [], []
    for i in range(R):
        th = i * (2.0 * math.pi / R)
        ux, uy = math.cos(th), math.sin(th)
        runs_against = ((ux * n[:, 0] + uy * n[:, 1]) < 1e-4) | ((ux * nn[:, 0] + uy * nn[:, 1]) < 1e-4)      # [E]
        tA, wA = A[:, 0] * ux + A[:, 1] * uy, -A[:, 0] * uy + A[:, 1] * ux
        tB, wB = B[:, 0] * ux + B[:, 1] * uy, -B[:, 0] * uy + B[:, 1] * ux
        tc = np.stack([x * ux + y * uy for x, y in corners])       # [4, ncell, 1]
        wc = np.stack([-x * uy + y * ux for x, y in corners])
        t0, t1, w0, w1 = tc.min(0), tc.max(0), wc.min(0), wc.max(0)
        a0, a1 = _clip_interval(tA[None, :], (tB - tA)[None, :], t0 - rs, t1 + L + rs)
        b0, b1 = _clip_interval(wA[None, :], (wB - wA)[None, :], w0 - rs, w1 + rs)
        l0, l1 = np.maximum(np.maximum(a0, b0), 0.0), np.minimum(np.minimum(a1, b1), 1.0)
        hit = (l0 <= l1) & in_front & runs_against[None, :]
        with np.errstate(invalid="ignore"):
            tmin = np.minimum(tA[None, :] + l0 * (tB - tA)[None, :], tA[None, :] + l1 * (tB - tA)[None, :])
        lb = np.maximum(np.maximum(tmin - rs - t1, lb_euclid), 0.0)
        hit &= lb < L
        c_idx, e_idx = np.nonzero(hit)
        cells_all.append(c_idx.astype(np.int64))
        rays_all.append(np.full(len(c_idx), i, np.int64))
        lbs_all.append(np.clip(np.floor(lb[c_idx, e_idx] * RAY_LIST_LB_SCALE) - 1.0, 0, 65535).astype(np.int64))
        edges_all.append(e_idx.astype(np.int64))
        raw_all.append(lb[c_idx, e_idx])
    cells_all, rays_all = np.concatenate(cells_all), np.concatenate(rays_all)
    lbs_all, edges_all, raw_all = np.concatenate(lbs_all), np.concatenate(edges_all), np.concatenate(raw_all)
    key = cells_all * R + rays_all
    order = np.lexsort((edges_all, lbs_all, key))
    ent = ((lbs_all[order] << 16) | edges_all[order]).astype(np.uint32)
    off = np.zeros(ncell * R + 1, np.int64)
    np.cumsum(np.bincount(key, minlength=ncell * R), out=off[1:])
    if return_bounds:
        return off.astype(np.int32), ent, raw_all[order]
    return off.astype(np.int32), ent


def compile_map(m: Map, *, cell: Optional[float] = None,
                contact_reach: float = 6.0, slack: float = 0.05, name: Optional[str] = None,
                spawn_override: Optional[Dict[str, List[dict]]] = None, view_range: float = 402.0) -> CompiledMap:
    """Blocks -> convex hulls -> flat arrays + uniform grid cell lists.

    ``contact_reach`` = agent radius + wall radius (contact iff centre-to-hull distance <= 6, SURVEY.md A.5),
    also the spawn rejection distance (``point_query_nearest(pos, 5)`` against hulls of radius 1 -> raw
    distance < 6) and what the "ray starts inside a wall's reach" lookup needs; ``slack`` is added so a point
    binned in fp32 can never miss a listed hull.  ``view_range`` = ray length + wall radius + ray radius: the
    reach the per-cell sensor candidate lists (``view_lists``) are built for.

    ``spawn_override`` maps agent id -> list of ``{"x","y","w","h"}`` regions and replaces what the
    map file says (used for the synthetic free-space spawns of the agh-map/labyrinth benchmarks).
    """
    hulls = [convex_hull_ccw(ring) for ring in m.blocks]
    hulls = _morton_sorted(hulls)      # spatially compact edge batches (the kernel culls 32 edges at a time)
    H = len(hulls)
    hull_off = np.zeros(H + 1, np.int32)
    for h, hv in enumerate(hulls):
        hull_off[h + 1] = hull_off[h] + len(hv)
    vert = np.concatenate(hulls, axis=0)
    normal = np.zeros_like(vert)
    edge_len = np.zeros(len(vert))
    hull_bb = np.zeros((H, 4))
    for h, hv in enumerate(hulls):
        prev = np.roll(hv, 1, axis=0)
        e = hv - prev
        ln = np.hypot(e[:, 0], e[:, 1])
        o = hull_off[h]
        normal[o:o + len(hv), 0] = e[:, 1] / ln      # rperp(e) = (e.y, -e.x)
        normal[o:o + len(hv), 1] = -e[:, 0] / ln
        edge_len[o:o + len(hv)] = ln
        hull_bb[h] = (hv[:, 0].min(), hv[:, 1].min(), hv[:, 0].max(), hv[:, 1].max())

    ids = [f"cop_{i}" for i in range(m.cops_count)] + [f"thief_{i}" for i in range(m.thieves_count)]
    init_pos = np.asarray(list(m.cops_positions) + list(m.thieves_positions), np.float64).reshape(-1, 2)
    region_off = [0]
    regions: List[Tuple[float, float, float, float]] = []
    src = dict(m.agent_spawn_regions)
    if spawn_override:
        src.update(spawn_override)
    for aid in ids:
        for r in src.get(aid, []) or []:
            regions.append((float(r["x"]), float(r["y"]), float(r["w"]), float(r["h"])))
        region_off.append(len(regions))

    if cell is None:
        cell = choose_cell_size(hull_bb, H)
    margin = contact_reach + slack + 2.0
    gx0 = float(hull_bb[:, 0].min() - margin)
    gy0 = float(hull_bb[:, 1].min() - margin)
    gx1 = float(hull_bb[:, 2].max() + margin)
    gy1 = float(hull_bb[:, 3].max() + margin)
    nx = max(1, int(math.ceil((gx1 - gx0) / cell)))
    ny = max(1, int(math.ceil((gy1 - gy0) / cell)))

    def build_lists(rho: float):
        per_cell: List[List[int]] = [[] for _ in range(nx * ny)]
        for h in range(H):
            o, e = hull_off[h], hull_off[h + 1]
            for c in _cells_touching_hull(vert[o:e], normal[o:e], hull_bb[h], rho, gx0, gy0, cell, nx, ny):
                per_cell[int(c)].append(h)   # ascending hull id by construction
        off = np.zeros(nx * ny + 1, np.int32)
        for c, lst in enumerate(per_cell):
            off[c + 1] = off[c] + len(lst)
        flat = np.asarray([h for lst in per_cell for h in lst], np.int32)
        return off, flat

    con_off, con_list = build_lists(contact_reach + slack)

    edge_hull = np.zeros(len(vert), np.int32)
    for h in range(H):
        edge_hull[int(hull_off[h]):int(hull_off[h + 1])] = h

    # candidate lists for the sensor sweep (view_range = ray length + wall radius + ray radius by default)
    view_off, view_edges = view_lists(vert, normal, hull_off, gx0, gy0, float(cell), nx, ny, float(view_range))

    return CompiledMap(
        name=name or Path(m.map_path).name.split(".")[0],
        window=tuple(float(v) for v in m.window_dimensions),
        n_cops=m.cops_count, n_thieves=m.thieves_count,
        hull_off=hull_off, vert=vert, normal=normal, edge_len=edge_len, hull_bb=hull_bb,
        init_pos=init_pos, region_off=np.asarray(region_off, np.int32),
        regions=np.asarray(regions, np.float64).reshape(-1, 4),
        grid_x0=gx0, grid_y0=gy0, cell=float(cell), nx=nx, ny=ny,
        edge_hull=edge_hull,
        con_cell_off=con_off, con_cell_hulls=con_list,
        view_cell_off=view_off, view_cell_edges=view_edges, view_range=float(view_range),
    )


def free_space_regions(m: Map, margin: float = 10.0) -> Dict[str, List[dict]]:
    """One spawn region per agent covering the hull bounding box (shrunk by ``margin``).

    The reference's own spawn rule (20 rejection-sampled tries, ``base_env.py:151-158``) then
    places agents in free space.  Used for agh-map / labyrinth, which define no regions.
    """
    xs = [v[0] for ring in m.blocks for v in ring]
    ys = [v[1] for ring in m.blocks for v in ring]
    reg = dict(x=min(xs) + margin, y=min(ys) + margin,
               w=max(xs) - min(xs) - 2 * margin, h=max(ys) - min(ys) - 2 * margin)
    ids = [f"cop_{i}" for i in range(m.cops_count)] + [f"thief_{i}" for i in range(m.thieves_count)]
    return {aid: [dict(reg)] for aid in ids}


#: agents injected into labyrinth.json (which ships none): 2 cops + 1 thief, default positions
#: in free cells of the scaled map; benchmark spawns come from ``free_space_regions``.
LABYRINTH_SCALE = (1280.0 / 30.0, 720.0 / 20.0)
LABYRINTH_AGENTS = [
    {"type": "cop", "x": 1.5 * LABYRINTH_SCALE[0], "y": 1.5 * LABYRINTH_SCALE[1]},
    {"type": "thief", "x": 24.5 * LABYRINTH_SCALE[0], "y": 10.5 * LABYRINTH_SCALE[1]},
    {"type": "cop", "x": 1.5 * LABYRINTH_SCALE[0], "y": 10.5 * LABYRINTH_SCALE[1]},
]


#: the maps shipped under maps_data/
SHIPPED_MAPS = ("squarinth", "labyrinth", "lbirinth", "grandbyrinth", "agh-map")


def load_named_map(name: str) -> Map:
    """Built-in maps by the names BASELINE.json uses; labyrinth gets its scale + injected agents."""
    if name == "labyrinth":
        return Map(builtin_map_path(name), scale=LABYRINTH_SCALE, agents=LABYRINTH_AGENTS)
    return Map(builtin_map_path(name))


# ---------------------------------------------------------------------------------- procedural maps
#: clearance of a maze's spawn regions from every wall hull beyond agent radius + wall radius
MAZE_SPAWN_MARGIN = 2.0


def generate_maze(seed: int, *, cols: int = 16, rows: int = 9, window: Tuple[float, float] = (1280.0, 720.0),
                  corridor: float = 60.0, wall: float = 16.0, n_cops: int = 2, n_thieves: int = 1,
                  agent_radius: float = 5.0, margin: float = MAZE_SPAWN_MARGIN) -> Map:
    """A perfect maze (exactly one path between any two cells) on a ``cols`` x ``rows`` grid, as a ``Map`` named
    ``maze-<seed>``.  The same seed gives the same maze on every host and rank (numpy's PCG64 stream).

    Cells are ``corridor`` units wide and separated by walls ``wall`` units thick; the maze is centred in ``window``.  Each
    straight run of wall segments along a grid line is one axis-aligned rect block (the outer boundary is four of them),
    so the map has few hulls and edges.  The cops spawn in one cell and the thieves in another, the two ends of a longest
    path of the maze; each spawn region keeps ``agent_radius + WALL_RADIUS + margin`` from every hull."""
    pitch = corridor + wall
    width, height = cols * pitch + wall, rows * pitch + wall
    if cols < 2 or rows < 2 or corridor <= 0 or wall <= 0:
        raise ValueError("a maze needs cols, rows >= 2 and positive corridor and wall widths")
    if width > window[0] or height > window[1]:
        raise ValueError(f"a {cols} x {rows} maze of pitch {pitch} ({width} x {height}) does not fit the window {window}")
    clear = agent_radius + WALL_RADIUS + margin
    if corridor <= 2 * clear:
        raise ValueError(f"corridor {corridor} leaves no spawn region at clearance {clear}")
    x0, y0 = (window[0] - width) / 2.0, (window[1] - height) / 2.0
    rng = np.random.default_rng(int(seed))
    # recursive backtracker over the cells; open_e[c, r]: passage (c, r) <-> (c + 1, r), open_n: (c, r) <-> (c, r + 1)
    open_e = np.zeros((cols, rows), bool)
    open_n = np.zeros((cols, rows), bool)
    seen = np.zeros((cols, rows), bool)
    stack = [(int(rng.integers(cols)), int(rng.integers(rows)))]
    seen[stack[0]] = True
    while stack:
        c, r = stack[-1]
        nbrs = [(dc, dr) for dc, dr in ((1, 0), (-1, 0), (0, 1), (0, -1))
                if 0 <= c + dc < cols and 0 <= r + dr < rows and not seen[c + dc, r + dr]]
        if not nbrs:
            stack.pop()
            continue
        dc, dr = nbrs[int(rng.integers(len(nbrs)))]
        if dc:
            open_e[min(c, c + dc), r] = True
        else:
            open_n[c, min(r, r + dr)] = True
        seen[c + dc, r + dr] = True
        stack.append((c + dc, r + dr))

    blocks: List[List[Tuple[float, float]]] = []

    def rect(x, y, w, h):
        blocks.append([(x, y), (x + w, y), (x + w, y + h), (x, y + h), (x, y)])

    # horizontal grid line j: segment i (under cell (i, j)) is a wall unless the cells (i, j - 1) and (i, j) connect
    for j in range(rows + 1):
        seg = [j in (0, rows) or not open_n[i, j - 1] for i in range(cols)]
        i = 0
        while i < cols:
            if not seg[i]:
                i += 1
                continue
            k = i
            while k + 1 < cols and seg[k + 1]:
                k += 1
            rect(x0 + i * pitch, y0 + j * pitch, (k - i + 1) * pitch + wall, wall)
            i = k + 1
    # vertical grid line i: segment j is a wall unless the cells (i - 1, j) and (i, j) connect
    for i in range(cols + 1):
        seg = [i in (0, cols) or not open_e[i - 1, j] for j in range(rows)]
        j = 0
        while j < rows:
            if not seg[j]:
                j += 1
                continue
            k = j
            while k + 1 < rows and seg[k + 1]:
                k += 1
            rect(x0 + i * pitch, y0 + j * pitch, wall, (k - j + 1) * pitch + wall)
            j = k + 1

    def farthest(start):
        dist = {start: 0}
        queue = [start]
        for c, r in queue:
            for nc, nr, ok in ((c + 1, r, c + 1 < cols and open_e[c, r]), (c - 1, r, c > 0 and open_e[c - 1, r]),
                               (c, r + 1, r + 1 < rows and open_n[c, r]), (c, r - 1, r > 0 and open_n[c, r - 1])):
                if ok and (nc, nr) not in dist:
                    dist[(nc, nr)] = dist[(c, r)] + 1
                    queue.append((nc, nr))
        return queue[-1]          # BFS order: the last cell reached is a farthest one
    cop_cell = farthest((0, 0))
    thief_cell = farthest(cop_cell)

    def region(cell):
        c, r = cell
        return dict(x=x0 + c * pitch + wall + clear, y=y0 + r * pitch + wall + clear,
                    w=corridor - 2 * clear, h=corridor - 2 * clear)

    def centre(cell):
        c, r = cell
        return x0 + c * pitch + wall + corridor / 2.0, y0 + r * pitch + wall + corridor / 2.0
    agents = []
    for kind, n, cell in (("cop", n_cops, cop_cell), ("thief", n_thieves, thief_cell)):
        cy = centre(cell)[1]
        reg = region(cell)
        for a in range(n):   # distinct start positions inside the cell's spawn region, spread along x
            px = reg["x"] + reg["w"] * (a + 1) / (n + 1)
            agents.append({"type": kind, "pos": [px, cy], "regions": [[reg["x"], reg["y"], reg["w"], reg["h"]]]})
    data = {"format": "catmap-1", "window": [float(window[0]), float(window[1])],
            "canvas": [float(window[0]), float(window[1])],
            "blocks": [[float(c) for v in ring for c in v] for ring in blocks], "agents": agents}
    return Map.from_dict(data, f"maze-{int(seed)}")
