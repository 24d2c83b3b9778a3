"""Pinball domain on B200: map loading and the batched env (K1), behind the same Python interface
as the CPU oracle (oracle/pinball.py PinballMap / PinballEnv - the stand-in for the reference,
which ships no code: /root/reference/README.md:1-2).

    env = PinballEnv("easy", batch=65536)
    state = env.reset()
    state, reward, done, hit_info = env.step(actions)

State lives in HBM as structure-of-arrays fp32 (x[B], y[B], vx[B], vy[B]); `step` accepts a CUDA
int32 tensor (no copies) or a NumPy array (host path: copies in and out through scg_step_host).
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import check, ptr

MAPS_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "maps")
N_ACTIONS = 5
FLAG_DONE, FLAG_KIND_SHIFT, FLAG_EDGE_SHIFT, FLAG_OBST_SHIFT = 1, 1, 8, 16


def unpack_flags(flags):
    """flags int32 (torch or numpy) -> (done, kind, obstacle, edge); obstacle/edge -1 without a hit."""
    if hasattr(flags, "is_cuda"):
        import torch
        done = (flags & FLAG_DONE) != 0
        kind = (flags >> FLAG_KIND_SHIFT) & 3
        neg = torch.full_like(flags, -1)
        edge = torch.where(kind != 0, (flags >> FLAG_EDGE_SHIFT) & 0xFF, neg)
        obst = torch.where(kind != 0, (flags >> FLAG_OBST_SHIFT) & 0xFFF, neg)
        return done, kind, obst, edge
    flags = np.asarray(flags, dtype=np.int32)
    done = (flags & FLAG_DONE) != 0
    kind = (flags >> FLAG_KIND_SHIFT) & 3
    edge = np.where(kind != 0, (flags >> FLAG_EDGE_SHIFT) & 0xFF, -1).astype(np.int32)
    obst = np.where(kind != 0, (flags >> FLAG_OBST_SHIFT) & 0xFFF, -1).astype(np.int32)
    return done, kind, obst, edge


class PinballMap:
    """A parsed map plus its device-resident edge table and broad-phase grid (scg_map_create)."""

    def __init__(self, ball_r, target, starts, polygons, grid_n=0):
        self.ball_r = float(ball_r)
        self.target = tuple(float(v) for v in target)
        self.starts = np.ascontiguousarray(np.asarray(starts, dtype=np.float32).reshape(-1, 2))
        self.polygons = [np.asarray(p, dtype=np.float32).reshape(-1, 2) for p in polygons]
        if len(self.starts) == 0:
            raise ValueError("map has no start position")
        verts = np.ascontiguousarray(np.concatenate(self.polygons, axis=0), dtype=np.float32)
        offs = np.zeros(len(self.polygons) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(p) for p in self.polygons])
        self._handle = C.c_void_p()
        lib = _lib.load()
        check(lib.scg_map_create(ptr(verts), ptr(offs), len(self.polygons), self.ball_r, self.target[0],
                                 self.target[1], self.target[2], ptr(self.starts), len(self.starts),
                                 int(grid_n), C.byref(self._handle)))     # grid_n 0: the library default (64)
        self.n_edges = lib.scg_map_num_edges(self._handle)
        self.n_candidates = lib.scg_map_num_candidates(self._handle)

    @property
    def handle(self):
        return self._handle

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.load().scg_map_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    @classmethod
    def from_file(cls, path, grid_n=0):
        ball, target, starts, polys = None, None, [], []
        with open(path) as f:
            for line in f:
                tok = line.split("#")[0].split()
                if not tok:
                    continue
                v = [float(u) for u in tok[1:]]
                if tok[0] == "ball":
                    ball = v[0]
                elif tok[0] == "target":
                    target = v[:3]
                elif tok[0] == "start":
                    starts = list(zip(v[0::2], v[1::2]))
                elif tok[0] == "polygon":
                    polys.append(list(zip(v[0::2], v[1::2])))
                else:
                    raise ValueError(f"unknown map directive {tok[0]!r}")
        if ball is None or target is None:
            raise ValueError("map needs 'ball' and 'target' lines")
        return cls(ball, target, starts, polys, grid_n)

    @classmethod
    def from_name(cls, name, grid_n=0):
        return cls.from_file(os.path.join(MAPS_DIR, name + ".cfg"), grid_n)

    def edge_table(self):
        """(edges float32 (E, 8), obstacle int32 (E,), local int32 (E,)) as the kernel uses them."""
        E = self.n_edges
        edges = np.empty((E, 8), dtype=np.float32)
        obst = np.empty(E, dtype=np.int32)
        local = np.empty(E, dtype=np.int32)
        check(_lib.load().scg_map_edge_table(self._handle, ptr(edges), ptr(obst), ptr(local)))
        return edges, obst, local

    def grid(self):
        """(G, cell_start int32 (G*G+1,), candidates int32) of the broad phase."""
        g = C.c_int()
        lib = _lib.load()
        check(lib.scg_map_grid(self._handle, C.byref(g), None, None))
        G = g.value
        cs = np.empty(G * G + 1, dtype=np.int32)
        cand = np.empty(max(self.n_candidates, 1), dtype=np.int32)
        check(lib.scg_map_grid(self._handle, C.byref(g), ptr(cs), ptr(cand)))
        return G, cs, cand[: self.n_candidates]

    def in_free_space(self, x, y, clearance=None):
        """True where a ball centre (x, y) is inside the unit square, outside every polygon and farther than
        `clearance` (default 1.05 ball radii) from every edge (fp64 geometry, host side)."""
        x = np.asarray(x, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64)
        c = self.ball_r * 1.05 if clearance is None else clearance
        ok = (x > 0) & (x < 1) & (y > 0) & (y < 1)
        for poly in self.polygons:
            p = poly.astype(np.float64)
            inside = np.zeros(x.shape, dtype=bool)
            for i in range(len(p)):
                (x1, y1), (x2, y2) = p[i], p[(i + 1) % len(p)]
                if y1 != y2:
                    inside ^= ((y1 > y) != (y2 > y)) & (x < (x2 - x1) * (y - y1) / (y2 - y1) + x1)
                dx, dy = x2 - x1, y2 - y1
                t = np.clip(((x - x1) * dx + (y - y1) * dy) / (dx * dx + dy * dy), 0, 1)
                ok &= np.hypot(x1 + t * dx - x, y1 + t * dy - y) > c
            ok &= ~inside
        return ok

    def validate(self):
        """Map sanity checks (SURVEY.md section 8f-4); returns a list of problems, empty when the map is sound."""
        problems = []
        if not 0.0 < self.ball_r < 0.1:
            problems.append(f"ball radius {self.ball_r} outside (0, 0.1)")
        tx, ty, tr = self.target
        if not (0 < tx < 1 and 0 < ty < 1 and tr > 0):
            problems.append("target outside the unit square or with non-positive radius")
        elif not bool(self.in_free_space(tx, ty, clearance=0.0)):
            problems.append("target centre lies inside an obstacle")
        for i, (sx, sy) in enumerate(self.starts):
            if not bool(self.in_free_space(float(sx), float(sy))):
                problems.append(f"start {i} ({sx:.3f}, {sy:.3f}) is not in free space")
        for i, poly in enumerate(self.polygons):
            if poly.min() < -1e-6 or poly.max() > 1 + 1e-6:
                problems.append(f"polygon {i} leaves the unit square")
            d = np.hypot(*(np.roll(poly, -1, axis=0) - poly).T)
            if d.min() < 1e-6:
                problems.append(f"polygon {i} has a degenerate edge")
            area2 = float(np.sum(poly[:, 0] * np.roll(poly[:, 1], -1) - np.roll(poly[:, 0], -1) * poly[:, 1]))
            if abs(area2) < 1e-9:
                problems.append(f"polygon {i} has zero area")
        # the border must be closed: a ball cannot sit on the edge of the unit square
        for x, y in ((0.001, 0.5), (0.999, 0.5), (0.5, 0.001), (0.5, 0.999)):
            if bool(self.in_free_space(x, y, clearance=0.0)):
                problems.append(f"no wall at the border near ({x}, {y}) (the bounds clamp would be reached)")
        return problems

    def sample_free_states(self, rng, n, vmax=1.0):
        """Synthetic benchmark inputs: positions uniform over free space (at least 1.05 ball radii
        from every obstacle, outside every polygon), velocities uniform in [-vmax, vmax]^2."""
        out = np.empty((n, 4), dtype=np.float32)
        k = 0
        c = self.ball_r * 1.05
        while k < n:
            m = max(2 * (n - k), 64)
            x = rng.uniform(0.0, 1.0, m)
            y = rng.uniform(0.0, 1.0, m)
            ok = np.ones(m, dtype=bool)
            for poly in self.polygons:
                p = poly.astype(np.float64)
                inside = np.zeros(m, dtype=bool)
                for i in range(len(p)):
                    (x1, y1), (x2, y2) = p[i], p[(i + 1) % len(p)]
                    if y1 != y2:
                        inside ^= ((y1 > y) != (y2 > y)) & (x < (x2 - x1) * (y - y1) / (y2 - y1) + x1)
                    dx, dy = x2 - x1, y2 - y1
                    t = np.clip(((x - x1) * dx + (y - y1) * dy) / (dx * dx + dy * dy), 0, 1)
                    ok &= np.hypot(x1 + t * dx - x, y1 + t * dy - y) > c
                ok &= ~inside
            x, y = x[ok][: n - k], y[ok][: n - k]
            out[k:k + len(x), 0] = x
            out[k:k + len(x), 1] = y
            k += len(x)
        out[:, 2:] = rng.uniform(-vmax, vmax, (n, 2)).astype(np.float32)
        return out


class PinballEnv:
    """Batched Pinball env on one GPU.  Same methods as oracle/pinball.py PinballEnv."""

    def __init__(self, pmap, batch=1, seed=0, env_offset=0, device=None, cull=True):
        import torch
        if not torch.cuda.is_available():
            raise _lib.ScgError("PinballEnv needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.map = pmap if isinstance(pmap, PinballMap) else PinballMap.from_name(pmap)
        self.batch = int(batch)
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        self.cull = bool(cull)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        B = self.batch
        self.soa = torch.zeros((4, B), dtype=torch.float32, device=self.device)   # x, y, vx, vy rows
        self.reward = torch.zeros(B, dtype=torch.float32, device=self.device)
        self.flags = torch.zeros(B, dtype=torch.int32, device=self.device)
        self.n_resets = 0
        self.reset()

    # -- views -----------------------------------------------------------------------------------
    @property
    def state(self):
        """(B, 4) view-by-copy of the SoA state, same orientation as the oracle's."""
        return self.soa.t().contiguous()

    def set_state(self, states):
        t = self.torch.as_tensor(np.asarray(states, dtype=np.float32)) if not hasattr(states, "is_cuda") else states
        self.soa.copy_(t.to(self.device, dtype=self.torch.float32).reshape(self.batch, 4).t())

    def reset(self, mask=None, states=None, step=None):
        torch = self.torch
        if states is not None:
            st = torch.as_tensor(np.asarray(states, dtype=np.float32)) if not hasattr(states, "is_cuda") else states
            st = st.to(self.device, dtype=torch.float32).reshape(self.batch, 4).t()
            if mask is None:
                self.soa.copy_(st)
            else:
                m = torch.as_tensor(np.asarray(mask)) if not hasattr(mask, "is_cuda") else mask
                m = m.to(self.device).bool()
                self.soa[:, m] = st[:, m]
        else:
            m8 = None
            if mask is not None:
                m = torch.as_tensor(np.asarray(mask)) if not hasattr(mask, "is_cuda") else mask
                if m.shape != (self.batch,):
                    raise ValueError("mask must have shape (B,)")
                m8 = m.to(self.device).to(torch.uint8).contiguous()
            key = self.n_resets if step is None else int(step)
            check(self.lib.scg_reset(self.map.handle, self.batch, ptr(m8), ptr(self.soa[0]), ptr(self.soa[1]),
                                     ptr(self.soa[2]), ptr(self.soa[3]), self.seed, key & 0xFFFFFFFF,
                                     self.env_offset, _lib.current_stream()))
        self.n_resets += 1
        return self.state

    def step(self, actions):
        """actions: CUDA int32 tensor (device path) or NumPy/host array (host path, copies included).
        Returns (state (B,4), reward (B,), done (B,), hit_info (B,3) = kind, obstacle, edge)."""
        torch = self.torch
        if not hasattr(actions, "is_cuda"):
            return self._step_host(np.asarray(actions))
        if actions.shape != (self.batch,):
            raise ValueError("actions must have shape (B,)")
        a = actions.to(self.device, dtype=torch.int32).contiguous()
        if self.batch and (int(a.min()) < 0 or int(a.max()) >= N_ACTIONS):
            raise ValueError("action out of range")
        s = self.soa
        check(self.lib.scg_step(self.map.handle, self.batch, ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(s[3]), ptr(a),
                                ptr(s[0]), ptr(s[1]), ptr(s[2]), ptr(s[3]), ptr(self.reward), ptr(self.flags),
                                int(self.cull), _lib.current_stream()))
        done, kind, obst, edge = unpack_flags(self.flags)
        return self.state, self.reward.clone(), done, torch.stack([kind, obst, edge], dim=1)

    def _step_host(self, actions):
        if actions.shape != (self.batch,):
            raise ValueError("actions must have shape (B,)")
        if self.batch and (actions.min() < 0 or actions.max() >= N_ACTIONS):
            raise ValueError("action out of range")
        a = np.ascontiguousarray(actions, dtype=np.int32)
        soa = self.soa.cpu().numpy()
        reward = np.empty(self.batch, dtype=np.float32)
        flags = np.empty(self.batch, dtype=np.int32)
        check(self.lib.scg_step_host(self.map.handle, self.batch, ptr(soa), ptr(a), ptr(reward), ptr(flags),
                                     _lib.current_stream()))
        self.soa.copy_(self.torch.from_numpy(soa))
        self.flags.copy_(self.torch.from_numpy(flags))
        done, kind, obst, edge = unpack_flags(flags)
        return np.ascontiguousarray(soa.T), reward, done, np.stack([kind, obst, edge], axis=1).astype(np.int32)
