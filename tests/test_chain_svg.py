"""tools/chain_svg.py without a GPU: the SVG of a map, initiation sets and synthetic trajectory records parses, has one
polygon per obstacle, breaks every path at an episode end and colours each option's segments with that option's
colour only."""
import os
import sys
import xml.etree.ElementTree as ET

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import chain_svg  # noqa: E402

NS = "{http://www.w3.org/2000/svg}"


class _Map:
    polygons = [np.array([[0.2, 0.2], [0.4, 0.2], [0.3, 0.4]], np.float32),
                np.array([[0.6, 0.6], [0.8, 0.6], [0.8, 0.8], [0.6, 0.8]], np.float32)]
    target = (0.9, 0.1, 0.04)
    starts = np.array([[0.1, 0.9], [0.2, 0.85]], np.float32)


def _records(rows):
    """rows: (step, env, x, y, option, term, episode_end) -> the dict trajectories() returns (other fields zero)."""
    a = np.array(rows, dtype=np.float64).reshape(-1, 7)
    n = len(a)
    state = np.zeros((n, 4), np.float32)
    state[:, :2] = a[:, 2:4]
    return dict(step=a[:, 0].astype(np.uint32), env=a[:, 1].astype(np.uint32), state=state,
                option=a[:, 4].astype(np.int32), action=np.zeros(n, np.int32), delta=np.zeros(n, np.float32),
                term=a[:, 5].astype(bool), label=np.zeros(n, bool), episode_end=a[:, 6].astype(bool),
                goal=np.zeros(n, bool), total=n)


def _walk(env, n, ends=(), switches=()):
    """n steps of one env along a line; option 0 then 1 after each index in `switches`; episode ends after `ends`."""
    rows, o = [], 0
    for t in range(n):
        term = t in ends or t in switches
        rows.append((t, env, 0.05 + 0.01 * t, 0.5 + 0.001 * env, o, term, t in ends))
        if t in switches:
            o = 1 - o
    return rows


def _parse(svg):
    root = ET.fromstring(svg)
    assert root.tag == NS + "svg"
    return root


def test_map_layers_and_one_polygon_per_obstacle():
    grid = np.zeros((3, 64, 64), bool)
    grid[0, 10:20, 5:30] = True
    grid[0, 12, 40:45] = True
    grid[2, :, :] = True
    root = _parse(chain_svg.render(_Map, _records(_walk(0, 10)), init_grid=grid, title="a <test> & map"))
    assert len(root.findall(f".//{NS}polygon")) == len(_Map.polygons)
    assert len(root.findall(f".//{NS}circle[@class='target']")) == 1
    assert len(root.findall(f".//{NS}rect[@class='start']")) == len(_Map.starts)
    groups = {g.get("data-option"): g for g in root.findall(f".//{NS}g[@class='initiation']")}
    assert set(groups) == {"0", "2"}                               # option 1's set is empty: nothing drawn
    assert len(groups["0"].findall(f"{NS}rect")) == 10 + 1          # one rect per horizontal run
    assert len(groups["2"].findall(f"{NS}rect")) == 64
    assert groups["0"].get("fill") == chain_svg.OPTION_COLORS[0] and groups["2"].get("fill") == chain_svg.OPTION_COLORS[2]


def test_paths_break_at_every_episode_end():
    ends = (3, 7, 12)
    tr = _records(_walk(5, 20, ends=ends) + _walk(6, 20))
    root = _parse(chain_svg.render(_Map, tr))
    lines = root.findall(f".//{NS}polyline")
    mine = [pl for pl in lines if pl.get("data-env") == "5"]
    assert len(mine) == len(ends) + 1
    assert len([pl for pl in lines if pl.get("data-env") == "6"]) == 1
    # no segment crosses an episode end: consecutive points of a polyline are consecutive steps of the walk
    xs = sorted(float(p.split(",")[0]) for pl in mine for p in pl.get("points").split())
    assert len(xs) == 20 and len(set(xs)) == 20
    marks = root.findall(f".//{NS}g[@class='terminations']/{NS}circle")
    assert len(marks) == len(ends)


def test_each_colour_belongs_to_one_option():
    tr = _records(_walk(0, 30, ends=(20,), switches=(4, 9, 14)) + _walk(1, 30, switches=(15,)))
    root = _parse(chain_svg.render(_Map, tr))
    lines = root.findall(f".//{NS}polyline")
    assert len(lines) == 5 + 2
    by_colour = {}
    for pl in lines:
        o = int(pl.get("data-option"))
        assert pl.get("stroke") == chain_svg.OPTION_COLORS[o]
        by_colour.setdefault(pl.get("stroke"), set()).add(o)
    assert all(len(v) == 1 for v in by_colour.values()) and len(by_colour) == 2
    # an option change keeps the path connected: the new option's line starts where the old one ended
    env0 = [pl.get("points").split() for pl in lines if pl.get("data-env") == "0"]
    for a, b in zip(env0[:3], env0[1:4]):
        assert a[-1] == b[0]


def test_empty_trajectory_renders():
    root = _parse(chain_svg.render(_Map, _records([])))
    assert root.findall(f".//{NS}polyline") == []
    assert len(root.findall(f".//{NS}polygon")) == len(_Map.polygons)
