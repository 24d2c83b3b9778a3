"""Host side of the trajectory log, without a GPU: the 32-byte record layout of include/scg_b200.h and the merge of
several ranks' logs by (step, env), with the merge the other device logs use."""
import numpy as np

from skill_chaining_with_graphs_b200.agent import TRAJECTORY_FLAGS, decode_trajectory_records, merge_episodes


def _records(step, env, state, action, option, flag_bits, delta):
    rec = np.zeros((len(step), 8), dtype=np.uint32)
    rec[:, 0], rec[:, 1] = step, env
    rec[:, 2:6] = np.asarray(state, dtype=np.float32).reshape(-1, 4).view(np.uint32)
    rec[:, 6] = (np.asarray(action, dtype=np.uint32) | (np.asarray(option, dtype=np.uint32) << 8) |
                 np.asarray(flag_bits, dtype=np.uint32))
    rec[:, 7] = np.asarray(delta, dtype=np.float32).view(np.uint32)
    return rec.view(np.int32)


def test_decode_every_flag_bit_alone_and_together():
    n = len(TRAJECTORY_FLAGS)
    bits = [0x10000 << i for i in range(n)] + [0, sum(0x10000 << i for i in range(n))]
    m = len(bits)
    rec = _records(np.arange(m) + 7, np.arange(m) + 1000, np.zeros((m, 4)), np.arange(m) % 5, np.arange(m) % 16,
                   bits, np.zeros(m))
    d = decode_trajectory_records(rec)
    assert d["step"].dtype == np.uint32 and d["env"].dtype == np.uint32
    assert d["action"].dtype == np.int32 and d["option"].dtype == np.int32
    assert np.array_equal(d["step"], np.arange(m) + 7) and np.array_equal(d["env"], np.arange(m) + 1000)
    assert np.array_equal(d["action"], np.arange(m) % 5) and np.array_equal(d["option"], np.arange(m) % 16)
    for i, k in enumerate(TRAJECTORY_FLAGS):
        want = np.zeros(m, dtype=bool)
        want[i] = want[m - 1] = True
        assert d[k].dtype == bool and np.array_equal(d[k], want), k


def test_state_and_delta_are_bit_exact():
    vals = np.array([0.1, -0.0, 1e-40, np.float32(np.pi), -3.0e38, np.inf, 0.999999, 2.0 ** -20], dtype=np.float32)
    state = np.stack([vals, vals[::-1], -vals, vals * 0.5], axis=1)
    nan = np.array([0x7FC01234], dtype=np.uint32).view(np.float32)[0]
    delta = np.concatenate([vals[:-1], [nan]]).astype(np.float32)
    rec = _records(np.zeros(8), np.zeros(8), state, np.zeros(8), np.zeros(8), np.zeros(8), delta)
    d = decode_trajectory_records(rec)
    assert d["state"].shape == (8, 4) and d["state"].dtype == np.float32
    assert np.array_equal(d["state"].view(np.uint32), state.view(np.uint32))
    assert np.array_equal(d["delta"].view(np.uint32), delta.view(np.uint32))


def test_ignores_the_unused_bits_of_word_6():
    rec = _records([3], [4], np.zeros((1, 4)), [4], [15], [0xFFF00000 | 0xF8 | 0x10000], [0.0])
    d = decode_trajectory_records(rec)
    assert int(d["action"][0]) == 4 and int(d["option"][0]) == 15
    assert d["term"][0] and not (d["label"][0] or d["episode_end"][0] or d["goal"][0])


def test_merge_ranks_by_step_then_env():
    a = decode_trajectory_records(_records([0, 0, 1, 1], [0, 2, 0, 2], np.arange(16).reshape(4, 4), [1, 2, 3, 4],
                                           [0, 1, 0, 1], [0, 0x10000, 0, 0x40000], [0.5, 1.5, 2.5, 3.5]))
    b = decode_trajectory_records(_records([0, 0, 1, 1], [5, 6, 5, 6], -np.arange(16).reshape(4, 4), [0, 0, 1, 1],
                                           [2, 2, 3, 3], [0x20000, 0, 0, 0x80000 | 0x40000], [9, 8, 7, 6]))
    a["total"], b["total"] = 4, 10
    m = merge_episodes([a, b])
    assert m["total"] == 14 and m["totals"] == [4, 10]
    assert np.array_equal(m["step"], [0, 0, 0, 0, 1, 1, 1, 1]) and np.array_equal(m["env"], [0, 2, 5, 6, 0, 2, 5, 6])
    assert m["state"].shape == (8, 4)
    assert np.array_equal(m["state"][2], -np.arange(4, dtype=np.float32)) and np.array_equal(m["state"][5], np.arange(12, 16))
    assert np.array_equal(m["delta"], np.array([0.5, 1.5, 9, 8, 2.5, 3.5, 7, 6], dtype=np.float32))
    assert np.array_equal(m["label"], [0, 0, 1, 0, 0, 0, 0, 0]) and np.array_equal(m["goal"], [0, 0, 0, 0, 0, 0, 0, 1])
    assert np.array_equal(m["episode_end"], [0, 0, 0, 0, 0, 1, 0, 1]) and np.array_equal(m["option"], [0, 1, 2, 2, 0, 1, 3, 3])
