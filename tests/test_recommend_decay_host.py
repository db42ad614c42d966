"""Host side of the freshness decay of top-K recommendation (no GPU): the pinned penalty arithmetic
(util.decay_penalty), the checks of recommend(decay=...) (util.check_decay), the request times of a split's sessions,
the --recommend_half_life_h flag and the ValueErrors the model raises before anything is uploaded."""
import datetime
import types

import numpy as np
import pytest

T0 = datetime.datetime(2017, 10, 1)
I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


def test_penalty_is_one_fp32_multiply_of_the_saturated_age():
    from tcar_b200._native import DECAY_MAX_AGE
    from tcar_b200.util import decay_penalty
    assert DECAY_MAX_AGE == 2 ** 23 - 1
    times = np.array([0, 10, 11, 12, I32_MIN, I32_MAX, -5], np.int64)
    p = decay_penalty([11, I32_MAX, I32_MIN], [0.1, 1.0, 3.0], times)
    assert p.dtype == np.float32 and p.shape == (3, 7)
    age = np.array([11, 1, 0, 0, DECAY_MAX_AGE, 0, 16], np.float32)     # a future article gets age 0
    assert (p[0] == np.float32(0.1) * age).all()
    assert p[1].tolist() == [DECAY_MAX_AGE] * 5 + [0, DECAY_MAX_AGE]      # ages saturate at 2^23 - 1
    assert (p[2] == 0).all()                                             # t_ref = INT32_MIN: nothing is older
    # the age is exact in float32 up to the bound: every integer below 2^24 is
    big = decay_penalty([DECAY_MAX_AGE], [1.0], [0, 1])
    assert big.tolist() == [[DECAY_MAX_AGE, DECAY_MAX_AGE - 1]]


def test_check_decay_layout_and_broadcast():
    from tcar_b200.util import check_decay
    out = check_decay(([5, -7, I32_MAX], 0.25), 3, [0, 100])
    assert out.dtype == np.int32 and out[:3].tolist() == [5, -7, I32_MAX]
    assert out[3:].view(np.float32).tolist() == [0.25] * 3
    out = check_decay((np.array([1, 2], np.uint16), np.array([0, 1e-3], np.float64)), 2, [0])
    assert out[2:].view(np.float32).tolist() == [0, np.float32(1e-3)]
    assert check_decay((np.zeros(0, np.int64), 1.0), 0, [0]).shape == (0,)
    # a large rate is fine while its largest penalty stays finite; the check uses the oldest item only
    check_decay(([10 ** 9], 1e30), 1, [10 ** 9 - 100])
    check_decay(([I32_MAX], 4e31), 1, [I32_MIN])                          # 4e31 x (2^23 - 1) < FLT_MAX


@pytest.mark.parametrize("decay,what", [
    (([0, 0], 0.1), "t_ref must hold B = 3"),
    (([0.0, 0.0, 0.0], 0.1), "t_ref must hold integers"),
    (([0, 2 ** 31, 0], 0.1), "session 1: decay t_ref 2147483648 outside int32"),
    (([0, 0, -2 ** 31 - 1], 0.1), "session 2"),
    (([0, 0, 0], [0.1, 0.2]), "one number or B = 3 numbers"),
    (([0, 0, 0], [[0.1, 0.2, 0.3]]), "one number or B = 3 numbers"),
    (([0, 0, 0], "fast"), "numbers"),
    (([0, 0, 0], [0.1, -0.5, 0.1]), "session 1: decay rate -0.5 is not finite and >= 0"),
    (([0, 0, 0], [0.1, 0.1, np.nan]), "session 2: decay rate nan"),
    (([0, 0, 0], np.inf), "session 0: decay rate inf"),
    (([0, 0, 0], 1e39), "session 0: decay rate 1e\\+39 overflows float32"),
    (([0, I32_MAX, 0], [0.1, 1e32, 0.1]), "session 1: .*penalty"),
    ((np.zeros(3, int),), "pair"),
    (np.zeros(3, int), "pair"),
])
def test_check_decay_refuses(decay, what):
    from tcar_b200.util import check_decay
    with pytest.raises(ValueError, match=what):
        check_decay(decay, 3, [I32_MIN, 0])


def test_session_request_times_are_the_window_ends():
    from tcar_b200.util import epoch_minutes, session_request_times, session_windows
    tdict = {"a": [{"click_t": T0}, {"click_t": T0 + datetime.timedelta(minutes=7, seconds=50)},
                   {"click_t": T0 + datetime.timedelta(hours=9)}],
             "b": [{"click_t": T0 + datetime.timedelta(days=1)}, {"click_t": T0 + datetime.timedelta(days=2)}]}
    t = session_request_times(["b", "a"], tdict)
    assert t.tolist() == epoch_minutes([T0 + datetime.timedelta(days=1), T0 + datetime.timedelta(minutes=7)]).tolist()
    lo, hi = session_windows(["b", "a"], tdict, 60)
    assert hi.tolist() == t.tolist() and (hi - lo).tolist() == [60, 60]


def test_half_life_flag():
    from tcar_b200.main import build_parser
    a = build_parser().parse_args(["--recommend_k", "20", "--recommend_half_life_h", "6"])
    assert a.recommend_half_life_h == 6.0
    a = build_parser().parse_args(["--recommend_k", "20", "--recommend_half_life_h", "6", "--recommend_max_age_h", "48",
                                   "--recommend_exclude_clicked"])
    assert (a.recommend_half_life_h, a.recommend_max_age_h, a.recommend_exclude_clicked) == (6.0, 48.0, True)
    assert build_parser().parse_args([]).recommend_half_life_h is None
    for bad in ("0", "-1", "x", "nan", "inf"):
        with pytest.raises(SystemExit):
            build_parser().parse_args(["--recommend_k", "20", "--recommend_half_life_h", bad])
    with pytest.raises(SystemExit):
        build_parser().parse_args(["--recommend_half_life_h", "6"])                      # requires --recommend_k
    with pytest.raises(SystemExit):
        build_parser().parse_args(["--recommend_k", "20", "--recommend_half_life_h", "6",
                                   "--recommend_max_per_category", "2"])


def test_model_checks_raise_before_anything_is_uploaded():
    """recommend(decay=...) raises its ValueError on the host (the GPU tests also count launches)."""
    from tcar_b200.model_combine import Seq2SeqAttNN
    m = Seq2SeqAttNN.__new__(Seq2SeqAttNN)
    m.N = 5
    bt = types.SimpleNamespace(B=2, T=3)
    with pytest.raises(ValueError, match="set_item_times"):
        m.recommend(bt, 5, decay=([0, 0], 0.1))
    m._item_time, m._item_time_min = object(), -100        # as if set: the decay checks come next
    for decay, what in [(([0, 0, 0], 0.1), "t_ref must hold B = 2"), (([0, 0], [0.1, -1.0]), "session 1: decay rate"),
                        (([0, I32_MAX], 1e33), "session 1: .*penalty")]:
        with pytest.raises(ValueError, match=what):
            m.recommend(bt, 5, decay=decay)
    m._iext_cat = object()
    for kw in ({"max_per_category": 2}, {"categories": ([0, 0, 0], [])}):
        with pytest.raises(ValueError, match="decay cannot be combined"):
            m.recommend(bt, 5, decay=([0, 0], 0.1), **kw)


def test_recommend_split_refuses_half_life_with_categories():
    from tcar_b200.model_combine import Seq2SeqAttNN
    m = Seq2SeqAttNN.__new__(Seq2SeqAttNN)
    with pytest.raises(ValueError, match="recommend_half_life_h"):
        m.recommend_split(None, None, {}, {"recommend_k": 20, "recommend_half_life_h": 6, "recommend_max_per_category": 2})
