"""Draw a learned skill chain as SVG, in pure Python: the map, each active option's initiation set and the greedy
trajectories of tracked envs coloured by the running option (the standard skill-chaining figure).

    svg = render(pmap, agent.trajectories(), init_grid=grid)
    open("chain.svg", "w").write(svg)

`pmap` needs `polygons` (list of (k, 2) vertex arrays), `target` (x, y, radius) and `starts` ((n, 2)), in the unit
square; both PinballMap classes have them.  `trajectories` is what SkillChainAgent.trajectories() returns (step, env,
state, option, term, episode_end; any order).  `init_grid` is an optional bool array (n_options, G, G): cell
[o, i, j] is True when option o's initiation set holds at x = (j + 0.5) / G, y = (i + 0.5) / G, zero velocity
(initiation_grid() builds it).  `occupancy` is an optional count array (n_options, G, G) indexed [option, iy, ix], what
SkillChainAgent.occupancy() returns as "counts": each option with any count gets a shaded layer of its visited cells,
darker on a log scale of the count, under the initiation sets, which are then drawn as outlines.  The picture has y
pointing up.
"""
from xml.sax.saxutils import escape

import numpy as np

# one colour per option slot (up to 16)
OPTION_COLORS = ("#1f77b4", "#ff7f0e", "#2ca02c", "#d62728", "#9467bd", "#8c564b", "#e377c2", "#17becf",
                 "#bcbd22", "#7f7f7f", "#393b79", "#637939", "#8c6d31", "#843c39", "#7b4173", "#3182bd")
SIZE = 640
OCCUPANCY_LEVELS = 8        # shades of an occupancy layer (log scale of the count)


def initiation_grid(options, active_mask, grid=64, device="cuda"):
    """(n_options, grid, grid) bool: options.initiation() at the cell centres, zero velocity, masked by the bits of
    `active_mask` (the controller's active_mask; inactive options come out all False)."""
    import torch
    c = (np.arange(grid, dtype=np.float32) + 0.5) / grid
    yy, xx = np.meshgrid(c, c, indexing="ij")
    s = np.zeros((grid * grid, 4), dtype=np.float32)
    s[:, 0], s[:, 1] = xx.ravel(), yy.ravel()
    inside = options.initiation(torch.as_tensor(s, device=device)).cpu().numpy().astype(bool)      # (n, K)
    active = np.array([(int(active_mask) >> k) & 1 for k in range(inside.shape[1])], dtype=bool)
    return (inside & active[None, :]).T.reshape(-1, grid, grid)


def _xy(x, y):
    return f"{float(x) * SIZE:.2f},{(1.0 - float(y)) * SIZE:.2f}"


def _runs(row):
    """[(start, length)] of the True runs of a bool row."""
    d = np.diff(np.concatenate([[0], row.astype(np.int8), [0]]))
    starts, ends = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
    return list(zip(starts.tolist(), (ends - starts).tolist()))


def _paths(tr):
    """Per env, in step order: (option, points) polylines and termination markers.  The segment s_t -> s_t+1 belongs to
    the option running at step t; a path breaks where an episode ended (s_t+1 is then a reset state) and starts a new
    polyline where the option changes.  A termination is marked where the execution ended: at s_t+1, or at s_t when
    the episode ended with it (the state reached before the reset is not logged)."""
    lines, marks = [], []
    env, step = np.asarray(tr["env"]), np.asarray(tr["step"]).astype(np.int64)
    for b in np.unique(env):
        idx = np.nonzero(env == b)[0]
        idx = idx[np.argsort(step[idx], kind="stable")]
        cur, pts = None, []
        for n, i in enumerate(idx):
            o, p = int(tr["option"][i]), tuple(tr["state"][i][:2])
            if cur is not None and o != cur:              # s_t ends the last segment of the previous option
                lines.append((int(b), cur, pts + [p]))
                pts = []
            cur = o
            pts.append(p)
            nxt = idx[n + 1] if n + 1 < len(idx) else None
            contiguous = nxt is not None and step[nxt] == step[i] + 1
            if tr["term"][i]:
                marks.append((int(b), o, p if tr["episode_end"][i] or not contiguous else tuple(tr["state"][nxt][:2])))
            if tr["episode_end"][i] or not contiguous:
                if len(pts) > 1:
                    lines.append((int(b), cur, pts))
                cur, pts = None, []
        if len(pts) > 1:
            lines.append((int(b), cur, pts))
    return lines, marks


def _outline(g, cw, ch):
    """SVG path data of the boundary of the True cells of a bool grid (row i from the bottom): one segment per cell edge
    between a True and a False cell."""
    p = np.pad(np.asarray(g, dtype=bool), 1)
    d = [f"M{j * cw:.2f},{SIZE - (i + 1) * ch:.2f}v{ch:.2f}" for i, j in zip(*np.nonzero(p[1:-1, 1:] != p[1:-1, :-1]))]
    d += [f"M{j * cw:.2f},{SIZE - i * ch:.2f}h{cw:.2f}" for i, j in zip(*np.nonzero(p[1:, 1:-1] != p[:-1, 1:-1]))]
    return "".join(d)


def _occupancy_layers(counts, color):
    """One <g class="occupancy"> per option with any count: its visited cells, shade level = ceil(L * log(1 + c) /
    log(1 + max c)) with the max over all options, so the layers compare; one <path> per level, a subpath per horizontal
    run of cells of that level."""
    c = np.asarray(counts, dtype=np.float64)
    out, top = [], np.log1p(c.max()) if c.size else 0.0
    cw, ch = SIZE / c.shape[2], SIZE / c.shape[1]
    for o in range(c.shape[0]):
        if not c[o].any():
            continue
        level = np.ceil(np.log1p(c[o]) / top * OCCUPANCY_LEVELS).astype(np.int64)
        out.append(f'<g class="occupancy" data-option="{o}" data-env-steps="{int(c[o].sum())}" fill="{color(o)}" '
                   'stroke="none">')
        for lv in range(1, OCCUPANCY_LEVELS + 1):
            d = [f"M{j0 * cw:g} {SIZE - (i + 1) * ch:g}h{n * cw:g}v{ch:g}h{-n * cw:g}z"
                 for i in range(c.shape[1]) for j0, n in _runs(level[i] == lv)]
            if d:
                out.append(f'<path data-level="{lv}" fill-opacity="{0.7 * lv / OCCUPANCY_LEVELS:.3f}" d="{"".join(d)}"/>')
        out.append('</g>')
    return out


def render(pmap, trajectories, init_grid=None, option_colors=OPTION_COLORS, title=None, occupancy=None):
    """-> the SVG document (str).  Layers, bottom to top: occupancy (one shaded layer per option, when given),
    initiation sets (translucent cells, horizontal runs merged into one rect; outlines over an occupancy layer),
    obstacles, target disc, start positions, trajectories (one polyline per run of one option), termination markers."""
    color = lambda o: option_colors[int(o) % len(option_colors)]
    out = [f'<svg xmlns="http://www.w3.org/2000/svg" width="{SIZE}" height="{SIZE}" viewBox="0 0 {SIZE} {SIZE}">',
           f'<rect x="0" y="0" width="{SIZE}" height="{SIZE}" fill="white" stroke="black"/>']
    if title:
        out.append(f'<title>{escape(str(title))}</title>')
    if occupancy is not None:
        out += _occupancy_layers(occupancy, color)
    if init_grid is not None:
        g = np.asarray(init_grid, dtype=bool)
        cell = SIZE / g.shape[2]
        for o in range(g.shape[0]):
            if not g[o].any():
                continue
            if occupancy is not None:
                out.append(f'<g class="initiation" data-option="{o}" fill="none" stroke="{color(o)}" stroke-width="1.5">'
                           f'<path d="{_outline(g[o], cell, SIZE / g.shape[1])}"/></g>')
                continue
            out.append(f'<g class="initiation" data-option="{o}" fill="{color(o)}" fill-opacity="0.18" stroke="none">')
            for i in range(g.shape[1]):
                y = SIZE - (i + 1) * (SIZE / g.shape[1])
                for j0, n in _runs(g[o, i]):
                    out.append(f'<rect x="{j0 * cell:.2f}" y="{y:.2f}" width="{n * cell:.2f}" '
                               f'height="{SIZE / g.shape[1]:.2f}"/>')
            out.append('</g>')
    out.append('<g class="obstacles" fill="#555555" stroke="black" stroke-width="0.5">')
    for poly in pmap.polygons:
        out.append('<polygon points="' + " ".join(_xy(x, y) for x, y in np.asarray(poly)) + '"/>')
    out.append('</g>')
    tx, ty, tr_ = (float(v) for v in pmap.target)
    cx, cy = _xy(tx, ty).split(",")
    out.append(f'<circle class="target" cx="{cx}" cy="{cy}" r="{tr_ * SIZE:.2f}" fill="#ffd700" stroke="black"/>')
    for x, y in np.asarray(pmap.starts).reshape(-1, 2):
        sx, sy = _xy(x, y).split(",")
        out.append(f'<rect class="start" x="{float(sx) - 4:.2f}" y="{float(sy) - 4:.2f}" width="8" height="8" '
                   f'fill="none" stroke="black" stroke-width="1.5"/>')
    lines, marks = _paths(trajectories)
    out.append('<g class="trajectories" fill="none" stroke-width="1.2" stroke-opacity="0.8">')
    for b, o, pts in lines:
        out.append(f'<polyline data-env="{b}" data-option="{o}" stroke="{color(o)}" points="' +
                   " ".join(_xy(x, y) for x, y in pts) + '"/>')
    out.append('</g>')
    out.append('<g class="terminations" stroke="black" stroke-width="0.4">')
    for b, o, (x, y) in marks:
        mx, my = _xy(x, y).split(",")
        out.append(f'<circle data-env="{b}" data-option="{o}" cx="{mx}" cy="{my}" r="2.5" fill="{color(o)}"/>')
    out.append('</g>')
    out.append('</svg>')
    return "\n".join(out) + "\n"
