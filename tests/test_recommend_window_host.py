"""Host side of the publish-time window of top-K recommendation (no GPU): epoch minutes, per-session windows from the
click log, label_outside counting, the --recommend_max_age_h flag and the ValueErrors of set_item_times / window=."""
import datetime
import random
import types

import numpy as np
import pytest

T0 = datetime.datetime(2017, 10, 1)


def test_epoch_minutes_floors_to_the_minute():
    from tcar_b200.util import epoch_minutes
    utc = datetime.timezone.utc
    got = epoch_minutes([datetime.datetime(1970, 1, 1), datetime.datetime(1970, 1, 1, 0, 1, 59),
                         datetime.datetime(1969, 12, 31, 23, 59, 30), T0,
                         datetime.datetime(2017, 10, 1, 2, 0, tzinfo=datetime.timezone(datetime.timedelta(hours=2)))])
    want = int((T0.replace(tzinfo=utc).timestamp()) // 60)
    assert got.tolist() == [0, 1, -1, want, want]
    assert got.dtype == np.int64


def time_dict_entry(clicks):
    return [{"click_t": c, "publish_t": T0, "delta_h": 1, "active_t": 1} for c in clicks]


def test_session_windows_use_the_last_input_click():
    from tcar_b200.util import epoch_minutes, session_windows
    tdict = {
        "a": time_dict_entry([T0 + datetime.timedelta(seconds=s) for s in (0, 70, 130, 9999)]),   # label click last
        "b": time_dict_entry([T0 + datetime.timedelta(minutes=5, seconds=59), T0 + datetime.timedelta(hours=3)]),
    }
    lo, hi = session_windows(["b", "a"], tdict, 24 * 60)
    t_req = epoch_minutes([T0 + datetime.timedelta(minutes=5), T0 + datetime.timedelta(minutes=2)])
    assert hi.tolist() == t_req.tolist()            # [-2]: the last INPUT click, seconds dropped
    assert (hi - lo).tolist() == [1440, 1440]


def test_session_windows_follow_each_ranks_batches():
    """Under torchrun every rank derives the windows of its own batches (Sampler.keep_rank_batches), in batch order."""
    from tcar_b200 import synth
    from tcar_b200.sampler import Sampler
    from tcar_b200.util import epoch_minutes, session_windows
    len_dict, sdict, tdict, _, _ = synth.make_sessions(300, 200, max_len=6, seed=5, train=False)
    world, per_rank = 3, []
    for rank in range(world):
        # every rank loads its own copy of the split and seeds alike (main.py), so all draw the same batches
        random.seed(2020)
        s = Sampler({L: list(keys) for L, keys in len_dict.items()}, sdict, tdict, batch_size=16, verbose=False)
        s.keep_rank_batches(rank, world)
        per_rank.append([(list(kb), session_windows(kb, tdict, 90)) for kb in s.session_id_batches])
    seen = set()
    for batches in per_rank:
        for kb, (lo, hi) in batches:
            assert len(lo) == len(hi) == len(kb)
            want = epoch_minutes([tdict[k][-2]["click_t"] for k in kb])
            assert (hi == want).all() and (lo == want - 90).all()
            assert not (set(kb) & seen)
            seen.update(kb)
    assert seen == set(sdict)


def test_count_outside():
    from tcar_b200.util import count_outside
    lo, hi = np.array([0, 10, 10, -5]), np.array([5, 10, 20, -1])
    assert count_outside([0, 10, 21, -6], lo, hi) == 2           # bounds inclusive
    assert count_outside([5, 9, 15, -1], lo, hi) == 1
    assert count_outside([], np.array([], int), np.array([], int)) == 0


def test_max_age_flag():
    from tcar_b200.main import build_parser
    a = build_parser().parse_args(["--recommend_k", "20", "--recommend_max_age_h", "1.5"])
    assert a.recommend_max_age_h == 1.5
    assert build_parser().parse_args([]).recommend_max_age_h is None
    for bad in ("0", "-2", "x", "nan"):
        with pytest.raises(SystemExit):
            build_parser().parse_args(["--recommend_k", "20", "--recommend_max_age_h", bad])
    with pytest.raises(SystemExit):
        build_parser().parse_args(["--recommend_max_age_h", "24"])          # requires --recommend_k


def test_item_time_checks():
    from tcar_b200.util import check_item_times
    assert check_item_times(np.array([0, -2 ** 31, 2 ** 31 - 1], np.int64), 3).dtype == np.int32
    assert check_item_times(np.arange(4, dtype=np.uint16), 4).tolist() == [0, 1, 2, 3]
    for times, what in [(np.arange(3), "N = 4"), (np.array([1, 2, 2 ** 31, 4]), "item 2: time 2147483648 outside int32"),
                        (np.array([0, -2 ** 31 - 1, 0, 0]), "item 1"), (np.zeros(4), "integers")]:
        with pytest.raises(ValueError, match=what):
            check_item_times(times, 4)


def test_window_checks():
    from tcar_b200.util import check_windows
    out = check_windows((np.array([1, 2, 3]), [1, 5, 2 ** 31 - 1]), 3)
    assert out.dtype == np.int32 and out.tolist() == [1, 2, 3, 1, 5, 2 ** 31 - 1]
    for window, what in [((np.arange(2), np.arange(3)), "lo must hold B = 3"),
                         ((np.arange(3), np.arange(4)), "hi must hold B = 3"),
                         ((np.array([0, 0, -2 ** 31 - 1]), np.zeros(3, int)), "session 2: window lo"),
                         ((np.zeros(3, int), np.array([0, 2 ** 31, 0])), "session 1: window hi 2147483648"),
                         ((np.array([0, 7, 9]), np.array([0, 6, 10])), "session 1: window lo 7 > hi 6"),
                         ((np.zeros(3), np.zeros(3)), "integers"),
                         (np.zeros(3, int), "pair")]:
        with pytest.raises(ValueError, match=what):
            check_windows(window, 3)


def test_model_checks_raise_before_anything_is_uploaded():
    """set_item_times / recommend(window=...) raise their ValueError on the host: no device buffer is touched (the
    GPU tests also count launches)."""
    from tcar_b200.model_combine import Seq2SeqAttNN
    m = Seq2SeqAttNN.__new__(Seq2SeqAttNN)
    m.N = 5
    for times, what in [([1, 2, 3], "N = 5"), ([0, 0, 0, 0, 2 ** 40], "item 4")]:
        with pytest.raises(ValueError, match=what):
            m.set_item_times(times)
    assert getattr(m, "_item_time", None) is None
    bt = types.SimpleNamespace(B=2, T=3)
    with pytest.raises(ValueError, match="set_item_times"):
        m.recommend(bt, 5, window=([0, 0], [1, 1]))
    m._item_time = object()                       # as if set: the window checks come next, still before any launch
    for window, what in [(([0, 0, 0], [1, 1]), "lo must hold B = 2"), (([0, 3], [1, 2]), "session 1: window lo 3")]:
        with pytest.raises(ValueError, match=what):
            m.recommend(bt, 5, window=window)
