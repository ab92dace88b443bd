"""Frames of swarms drawn on the device (`swarm_render`, include/swarm_b200.h), and the NumPy statement of its pixel rules.

    r = SwarmRenderer(sim, env_ids=[0, 5], width=512, height=512, trail_len=15)
    r.record()                        # after each step: the listed envs' positions go into the trail ring (a device copy)
    frames = r.render()               # uint8 CUDA tensor [2, 512, 512, 3], gym's rgb_array layout

`sim` is a BatchedAssemblySim or a BatchedFlockingSim.  A frame shows, bottom to top: the arena (white) and the area outside
it (grey), the env's target cells, each agent's trail, and the agents, coloured by whether the last observation found them
inside the shape.  The rules are DESIGN.md §10; `render_reference` states them in NumPy and the device frames equal its output
bit for bit.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import SwarmRenderArgs, check

CELLS, AGENTS, TRAILS = _lib.SWARM_RENDER_CELLS, _lib.SWARM_RENDER_AGENTS, _lib.SWARM_RENDER_TRAILS
ARENA, OUTSIDE, CELL, TRAIL, AGENT_IN, AGENT_OUT = range(6)      # palette rows (the SWARM_RGB_* order of the header)


def palette():
    """[6, 3] uint8: the library's colours, rows in the order ARENA, OUTSIDE, CELL, TRAIL, AGENT_IN, AGENT_OUT."""
    buf = (C.c_uint8 * 18)()
    n = _lib.load().swarm_render_palette(buf)
    return np.frombuffer(bytes(buf), dtype=np.uint8).reshape(n, 3).copy()


def render_reference(width, height, view, arena, p, size_a, *, in_flags=None, cells=None, in_thresh=0.0, trail=None,
                     half=(math.inf, math.inf), flags=CELLS | AGENTS | TRAILS, colours=None):
    """One frame by the rules of DESIGN.md §10, in float64 with every operation rounded separately.

    view, arena: (xmin, ymax, xmax, ymin); p: [2, n_a] positions; in_flags: [n_a] (None = every agent 'outside', a flocking
    handle); cells: [2, n_g] cell centres and in_thresh the env's in-shape threshold (disc rr = in_thresh * 0.5); trail:
    [L, 2, n_a] samples, oldest first; half: (half_w, half_h) of the arena (longer trail steps are periodic wraps).
    Returns uint8 [height, width, 3].

    Each primitive is evaluated on the pixels of its bounding box widened by two pixels, which contains every pixel it can
    cover; that is what makes this fast enough for tests, and it does not change a single pixel."""
    W, H = int(width), int(height)
    x0, y1, x1, y0 = (float(v) for v in view)
    sx, sy = (x1 - x0) / W, (y1 - y0) / H
    X = x0 + (np.arange(W, dtype=np.float64) + 0.5) * sx
    Y = y1 - (np.arange(H, dtype=np.float64) + 0.5) * sy
    ax0, ay1, ax1, ay0 = (float(v) for v in arena)
    lab = np.where(((ay0 <= Y) & (Y <= ay1))[:, None] & ((ax0 <= X) & (X <= ax1))[None, :], ARENA, OUTSIDE).astype(np.int8)

    def window(xlo, xhi, ylo, yhi):
        """pixel rows / columns whose centres can lie in [xlo, xhi] x [ylo, yhi]"""
        c0 = max(int(math.floor((xlo - x0) / sx - 0.5)) - 2, 0)
        c1 = min(int(math.ceil((xhi - x0) / sx - 0.5)) + 3, W)
        r0 = max(int(math.floor((y1 - yhi) / sy - 0.5)) - 2, 0)
        r1 = min(int(math.ceil((y1 - ylo) / sy - 0.5)) + 3, H)
        return slice(r0, max(r0, r1)), slice(c0, max(c0, c1))

    def disc(cx, cy, rr, value):
        r = math.sqrt(rr)
        if not (math.isfinite(cx) and math.isfinite(cy)):
            return
        rs, cs = window(cx - r, cx + r, cy - r, cy + r)
        dx = X[cs] - cx
        dy = Y[rs] - cy
        hit = (dx * dx)[None, :] + (dy * dy)[:, None] <= rr
        lab[rs, cs][hit] = value

    if (flags & CELLS) and cells is not None:
        rr = float(in_thresh) * 0.5
        for j in range(cells.shape[1]):
            disc(float(cells[0, j]), float(cells[1, j]), rr, CELL)
    if (flags & TRAILS) and trail is not None:
        w = size_a * 0.25
        ww = w * w
        for k in range(trail.shape[0] - 1):
            for i in range(trail.shape[2]):
                ax, ay, bx, by = (float(trail[k, 0, i]), float(trail[k, 1, i]), float(trail[k + 1, 0, i]), float(trail[k + 1, 1, i]))
                ux, uy = bx - ax, by - ay
                if not (abs(ux) <= half[0] and abs(uy) <= half[1]):
                    continue
                ll = ux * ux + uy * uy
                rs, cs = window(min(ax, bx) - w, max(ax, bx) + w, min(ay, by) - w, max(ay, by) + w)
                ex = ((X[cs] - ax) * ux)[None, :]
                ey = ((Y[rs] - ay) * uy)[:, None]
                t = (ex + ey) / ll if ll > 0 else np.zeros((rs.stop - rs.start, cs.stop - cs.start))
                t = np.minimum(np.maximum(t, 0.0), 1.0)
                dx = X[cs][None, :] - (ax + t * ux)
                dy = Y[rs][:, None] - (ay + t * uy)
                lab[rs, cs][dx * dx + dy * dy <= ww] = TRAIL
    if flags & AGENTS:
        rr = size_a * size_a
        for i in range(p.shape[1]):              # ascending index: where agents overlap, the largest index is painted last
            inside = in_flags is not None and (int(in_flags[i]) & 1)
            disc(float(p[0, i]), float(p[1, i]), rr, AGENT_IN if inside else AGENT_OUT)
    return (palette() if colours is None else colours)[lab]


class SwarmRenderer:
    """rgb_array frames of the envs `env_ids` of `sim` (duplicates allowed), `width` x `height` pixels of `view` =
    (xmin, ymax, xmax, ymin) (default: the arena), with trails of the last `trail_len` recorded positions."""

    def __init__(self, sim, env_ids, width, height, view=None, trail_len=0):
        self.sim, self.lib = sim, _lib.load()
        self.env_ids = np.ascontiguousarray(env_ids, dtype=np.int32).reshape(-1)
        self._ids_dev = torch.from_numpy(self.env_ids.astype(np.int64)).to(sim.device)
        self.width, self.height = int(width), int(height)
        self.view = (0.0, 0.0, 0.0, 0.0) if view is None else tuple(float(v) for v in view)
        self.frames = None
        count = self.env_ids.shape[0]
        self.trail_cap = int(trail_len)
        self.trail = (torch.zeros(self.trail_cap, count, 2, sim.n_a, dtype=torch.float64, device=sim.device)
                      if self.trail_cap > 0 else None)
        self.trail_len, self.trail_head = 0, max(self.trail_cap - 1, 0)

    def record(self):
        """Appends the envs' current positions to the trail ring (overwriting the oldest sample once it is full)."""
        if self.trail is None:
            return
        self.trail_head = (self.trail_head + 1) % self.trail_cap
        torch.index_select(self.sim.p, 0, self._ids_dev, out=self.trail[self.trail_head])
        self.trail_len = min(self.trail_len + 1, self.trail_cap)

    def clear(self):
        """Forgets the recorded trail."""
        self.trail_len = 0

    def render(self, cells=True, agents=True, trails=True):
        """uint8 CUDA tensor [count, height, width, 3]; the same tensor every call, overwritten by the next one."""
        if self.frames is None:
            self.frames = torch.empty(self.env_ids.shape[0], self.height, self.width, 3, dtype=torch.uint8, device=self.sim.device)
        a = SwarmRenderArgs()
        a.struct_size = C.sizeof(SwarmRenderArgs)
        a.width, a.height = self.width, self.height
        a.flags = (CELLS if cells else 0) | (AGENTS if agents else 0) | (TRAILS if trails else 0)
        a.count, a.env_ids = self.env_ids.shape[0], self.env_ids.ctypes.data
        a.view[:] = self.view
        if self.trail is not None:
            a.trail, a.trail_cap, a.trail_len, a.trail_head = self.trail.data_ptr(), self.trail_cap, self.trail_len, self.trail_head
        a.frames = self.frames.data_ptr()
        check(self.lib.swarm_render(self.sim._h, C.byref(a), self.sim._stream()), "swarm_render")
        return self.frames
