"""The occupancy grid without a GPU: the cell rule of tests/oracle_occupancy.py at its edges, the oracle helper counting
every env-step once by the option it ran and the state it began at, AgentConfig's check of the grid size, and the
occupancy layers of tools/chain_svg.py."""
import os
import sys
import xml.etree.ElementTree as ET

import numpy as np
import pytest

import oracle
from oracle_occupancy import OccupancyAgent, cells
from oracle_replay import activate, default_theta

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import chain_svg  # noqa: E402

NS = "{http://www.w3.org/2000/svg}"


@pytest.mark.parametrize("G", [1, 2, 16, 64, 128])
def test_cell_rule_known_answers(G):
    below = np.nextafter(np.float32(1.0 / G), np.float32(0.0), dtype=np.float32)    # largest fp32 below 1/G
    assert cells(np.float32(0.0), G) == 0
    assert cells(below, G) == 0
    assert cells(np.float32(1.0), G) == G - 1
    assert cells(np.float32(-1e-7), G) == 0
    assert cells(np.float32(-0.75), G) == 0
    assert cells(np.float32(1.5), G) == G - 1
    k = np.arange(G)
    assert np.array_equal(cells((k / G).astype(np.float32), G), k)                  # exactly k / G -> cell k
    if G > 1:
        assert np.array_equal(cells(np.nextafter((k[1:] / G).astype(np.float32), np.float32(0.0)), G), k[:-1])


def test_cell_rule_grid_of_one():
    v = np.array([-0.5, 0.0, 1e-30, 0.3, 0.999999, 1.0, 2.0], dtype=np.float32)
    assert not cells(v, 1).any()


def _agent(B=24, T=40, K=3, grid=16, **kw):
    cfg = dict(map="easy", batch=B, order=2, max_options=K, seed=7, epsilon=1.0, max_episode_steps=9, option_timeout=5,
               gestation_successes=3, example_capacity=1 << 12)
    cfg.update(kw)
    ag = OccupancyAgent(oracle.AgentConfig(**cfg), grid=grid)
    activate(ag, default_theta(K), K - 1)          # options 0 .. K-2 active, K-1 gestating
    states, opts = [], []
    for t in range(T):
        states.append(np.array(ag.env.state, dtype=np.float32, copy=True))
        opts.append(ag.option.copy())
        ag.step()
        if (t + 1) % 10 == 0:
            ag.manage()
    return ag, np.stack(states), np.stack(opts)


def test_oracle_counts_every_env_step_once():
    B, T, G = 24, 40, 16
    ag, S, O = _agent(B, T, grid=G)
    assert ag.counts.dtype == np.uint64 and ag.counts.shape == (3, G, G)
    assert int(ag.counts.sum()) == B * T
    # the same counts straight from the states and options before every step
    want = np.zeros_like(ag.counts)
    for s, o in zip(S, O):
        for b in range(B):
            want[o[b], cells(s[b, 1], G), cells(s[b, 0], G)] += 1
    assert np.array_equal(ag.counts, want)
    assert (ag.counts.reshape(3, -1).sum(axis=1) > 0).sum() >= 2          # more than one option ran
    assert ag.trajectory_log()["step"].size == 0                          # no tracked envs: the other logs still run


@pytest.mark.parametrize("G", [3, 256, -1, 0.5, 12, True])
def test_agent_config_rejects_bad_grid(G):
    import skill_chaining_with_graphs_b200 as scg
    with pytest.raises(ValueError):
        scg.AgentConfig(occupancy_grid=G)


def test_agent_config_accepts_every_power_of_two():
    import skill_chaining_with_graphs_b200 as scg
    assert scg.AgentConfig().occupancy_grid == 0
    for G in (1, 2, 4, 8, 16, 32, 64, 128):
        assert scg.AgentConfig(occupancy_grid=G).occupancy_grid == G


class _Map:
    polygons = [np.array([[0.2, 0.2], [0.4, 0.2], [0.3, 0.4]], np.float32)]
    target = (0.9, 0.1, 0.04)
    starts = np.array([[0.1, 0.9]], np.float32)


def _empty_records():
    z = np.zeros(0)
    return dict(step=z.astype(np.uint32), env=z.astype(np.uint32), state=np.zeros((0, 4), np.float32),
                option=z.astype(np.int32), term=z.astype(bool), episode_end=z.astype(bool), total=0)


def test_chain_svg_one_occupancy_layer_per_option_that_ran():
    G = 32
    counts = np.zeros((4, G, G), dtype=np.uint64)
    counts[0, 3, 4:9] = [1, 10, 100, 1000, 10 ** 6]
    counts[2, :, 20] = 7
    init = np.zeros((4, G, G), bool)
    init[0, 2:6, 3:10] = True
    init[1, 10:12, 10:12] = True
    svg = chain_svg.render(_Map, _empty_records(), init_grid=init, occupancy=counts, title="occupancy")
    root = ET.fromstring(svg)
    assert root.tag == NS + "svg"
    layers = root.findall(f".//{NS}g[@class='occupancy']")
    assert [g.get("data-option") for g in layers] == ["0", "2"]                     # option 1 and 3 never ran
    assert [int(g.get("data-env-steps")) for g in layers] == [int(counts[0].sum()), int(counts[2].sum())]
    for g in layers:
        assert g.get("fill") == chain_svg.OPTION_COLORS[int(g.get("data-option"))]
    # option 0: five cells of five different counts -> five shades, darker for more steps (log scale)
    paths = layers[0].findall(f"{NS}path")
    x = [float(p.get("d")[1:].split()[0]) for p in paths]
    op = [float(p.get("fill-opacity")) for p in paths]
    assert len(paths) == 5 and all(p.get("d").count("M") == 1 for p in paths)
    assert sorted(x) == [4 * 640 / G + k * 640 / G for k in range(5)]
    assert [o for _, o in sorted(zip(x, op))] == sorted(op) and len(set(op)) == 5 and op[-1] == pytest.approx(0.7)
    # option 2: one column of equal counts -> one level, one run per row
    paths = layers[1].findall(f"{NS}path")
    assert len(paths) == 1 and paths[0].get("d").count("M") == G
    # the initiation sets lie over the occupancy layers, as outlines
    kids = list(root)
    first_init = min(i for i, e in enumerate(kids) if e.get("class") == "initiation")
    assert max(i for i, e in enumerate(kids) if e.get("class") == "occupancy") < first_init
    outlines = root.findall(f".//{NS}g[@class='initiation']")
    assert [g.get("data-option") for g in outlines] == ["0", "1"] and all(g.get("fill") == "none" for g in outlines)
    d = outlines[1].find(f"{NS}path").get("d")
    assert d.count("M") == 8                                              # a 2 x 2 block has 8 unit edges

