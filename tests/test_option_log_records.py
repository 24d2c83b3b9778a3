"""Host side of the option log, without a GPU: the 32-byte record layout of include/scg_b200.h and the merge of several
ranks' logs by (step, env), with the same merge the episode log uses."""
import numpy as np

from skill_chaining_with_graphs_b200.agent import OPTION_OUTCOMES, decode_option_records, merge_episodes


def _records(step, env, option, outcome_bits, duration, start, end):
    rec = np.zeros((len(step), 8), dtype=np.uint32)
    rec[:, 0], rec[:, 1] = step, env
    rec[:, 2] = np.asarray(option, dtype=np.uint32) | np.asarray(outcome_bits, dtype=np.uint32)
    rec[:, 3] = np.asarray(duration, dtype=np.int32).view(np.uint32)
    rec[:, 4:6] = np.asarray(start, dtype=np.float32).reshape(-1, 2).view(np.uint32)
    rec[:, 6:8] = np.asarray(end, dtype=np.float32).reshape(-1, 2).view(np.uint32)
    return rec.view(np.int32)


def test_decode_record_layout_every_outcome_bit():
    n = len(OPTION_OUTCOMES)
    # record i has only outcome bit i set, the last one all of them, the one before none
    bits = [1 << (8 + i) for i in range(n)] + [0, 0x3F00]
    m = len(bits)
    step = np.arange(m, dtype=np.uint32) * 70001
    env = np.full(m, 0xFFFFFFF0, dtype=np.uint32) - np.arange(m, dtype=np.uint32)
    option = np.arange(m) % 16
    start = np.stack([np.linspace(0.01, 0.99, m), np.linspace(-0.5, 0.5, m)], axis=1).astype(np.float32)
    end = (start[:, ::-1] + np.float32(1e-7)).astype(np.float32)
    dur = np.arange(1, m + 1, dtype=np.int32) * 1000003
    d = decode_option_records(_records(step, env, option, bits, dur, start, end))
    assert d["step"].dtype == np.uint32 and d["step"].tolist() == step.tolist()
    assert d["env"].dtype == np.uint32 and d["env"].tolist() == env.tolist()
    assert d["option"].dtype == np.int32 and d["option"].tolist() == option.tolist()
    assert d["duration"].dtype == np.int32 and d["duration"].tolist() == dur.tolist()
    for i, k in enumerate(OPTION_OUTCOMES):
        assert d[k].dtype == bool
        want = [j == i or j == m - 1 for j in range(m)]
        assert d[k].tolist() == want, k
    assert d["start"].dtype == np.float32 and d["start"].shape == (m, 2)
    assert np.array_equal(d["start"].view(np.uint32), start.view(np.uint32))
    assert np.array_equal(d["end"].view(np.uint32), end.view(np.uint32))
    empty = decode_option_records(np.zeros((0, 8), dtype=np.int32))
    assert all(len(v) == 0 for v in empty.values()) and empty["start"].shape == (0, 2)


def test_merge_orders_by_step_then_env():
    a = decode_option_records(_records([1, 4, 4], [0, 1, 2], [0, 1, 2], [0x100, 0, 0x2400], [1, 2, 3],
                                       [[0.1, 0.2], [0.3, 0.4], [0.5, 0.6]], [[1.1, 1.2], [1.3, 1.4], [1.5, 1.6]]))
    b = decode_option_records(_records([0, 4, 9], [10, 11, 10], [3, 0, 1], [0x1000, 0x800, 0x300], [4, 5, 6],
                                       [[0.7, 0.8], [0.9, 1.0], [0.0, 0.1]], [[2.1, 2.2], [2.3, 2.4], [2.5, 2.6]]))
    a["total"], b["total"] = 7, 3
    m = merge_episodes([a, b])
    assert m["step"].tolist() == [0, 1, 4, 4, 4, 9] and m["env"].tolist() == [10, 0, 1, 2, 11, 10]
    assert m["option"].tolist() == [3, 0, 1, 2, 0, 1] and m["duration"].tolist() == [4, 1, 2, 3, 5, 6]
    assert m["hit"].tolist() == [False, True, False, False, False, True]
    assert m["label"].tolist() == [False, False, False, False, False, True]
    assert m["left"].tolist() == [True, False, False, False, False, False]
    assert m["option_timeout"].tolist() == [False, False, False, False, True, False]
    assert m["env_done"].tolist() == [False, False, False, True, False, False]
    assert m["episode_timeout"].tolist() == [False, False, False, True, False, False]
    assert np.allclose(m["start"][:, 0], [0.7, 0.1, 0.3, 0.5, 0.9, 0.0])
    assert np.allclose(m["end"][:, 1], [2.2, 1.2, 1.4, 1.6, 2.4, 2.6]) and m["end"].shape == (6, 2)
    assert m["total"] == 10 and m["totals"] == [7, 3]
    assert set(m) == set(a) | {"totals"}
