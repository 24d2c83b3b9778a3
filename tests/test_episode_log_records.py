"""Host side of the episode log, without a GPU: the 16-byte record layout of include/scg_b200.h and the merge of
several ranks' logs by (step, env)."""
import numpy as np

from skill_chaining_with_graphs_b200.agent import decode_episode_records, merge_episodes


def _records(step, env, ret, length, goal):
    rec = np.zeros((len(step), 4), dtype=np.uint32)
    rec[:, 0], rec[:, 1] = step, env
    rec[:, 2] = np.asarray(ret, dtype=np.float32).view(np.uint32)
    rec[:, 3] = np.asarray(length, dtype=np.uint32) | (np.asarray(goal, dtype=np.uint32) << 31)
    return rec.view(np.int32)


def test_decode_record_layout():
    rec = _records([3, 3, 70000], [5, 9, 0xFFFFFFF0], [-14.0, 9993.0, -2e6], [14, 7, 0x7FFFFFFF], [0, 1, 1])
    d = decode_episode_records(rec)
    assert d["step"].dtype == np.uint32 and d["step"].tolist() == [3, 3, 70000]
    assert d["env"].tolist() == [5, 9, 0xFFFFFFF0]
    assert d["ret"].dtype == np.float32 and d["ret"].tolist() == [-14.0, 9993.0, -2e6]
    assert d["length"].dtype == np.int32 and d["length"].tolist() == [14, 7, 0x7FFFFFFF]
    assert d["goal"].tolist() == [False, True, True]
    empty = decode_episode_records(np.zeros((0, 4), dtype=np.int32))
    assert all(len(v) == 0 for v in empty.values())


def test_merge_orders_by_step_then_env():
    a = decode_episode_records(_records([1, 4, 4], [0, 1, 2], [-1, -2, -3], [1, 2, 3], [0, 0, 1]))
    b = decode_episode_records(_records([0, 4, 9], [10, 11, 10], [-4, -5, -6], [4, 5, 6], [1, 0, 0]))
    a["total"], b["total"] = 7, 3
    m = merge_episodes([a, b])
    assert m["step"].tolist() == [0, 1, 4, 4, 4, 9] and m["env"].tolist() == [10, 0, 1, 2, 11, 10]
    assert m["ret"].tolist() == [-4, -1, -2, -3, -5, -6] and m["length"].tolist() == [4, 1, 2, 3, 5, 6]
    assert m["goal"].tolist() == [True, False, False, True, False, False]
    assert m["total"] == 10 and m["totals"] == [7, 3]
