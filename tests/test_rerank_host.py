"""Host side of impression-list ranking (no GPU): candidate lists, the MIND metric definitions, the CLI flag."""
import math

import numpy as np


def test_impression_candidates_map_dedup_and_append_the_label():
    from tcar_b200.sampler import impression_candidates
    item_dict = {"a%d" % i: i + 1 for i in range(10)}
    impressions = {
        0: ["a3", "x1", "a5", "a3", "a7"],       # unknown article dropped, repeat dropped (first kept), label appended
        1: ["a2", "a4", "a2"],                   # label already listed: kept in place, not appended again
        5: ["x9"],                               # only unknown articles -> [label]
    }
    keys = ["0_4", 1, 3, "5_2"]                   # train-style "<sid>_<len>" keys and plain test keys; 3 has no list
    labels = [9, 4, 6, 1]
    off, ids = impression_candidates(keys, labels, impressions, item_dict)
    assert off.dtype == np.int32 and ids.dtype == np.int32
    lists = [ids[off[b]:off[b + 1]].tolist() for b in range(len(keys))]
    assert lists == [[3, 5, 7, 9], [2, 4], [6], [1]]
    assert off.tolist() == [0, 4, 6, 7, 8]


def test_impression_candidates_empty_batch():
    from tcar_b200.sampler import impression_candidates
    off, ids = impression_candidates([], [], {}, {})
    assert off.tolist() == [0] and ids.size == 0


def test_impression_metrics_hand_worked():
    from tcar_b200.util import impression_metrics, impression_sums
    rank = [1, 3, 6, 12, 2]
    auc = [1.0, 0.75, 0.5, 0.25, 0.9]
    n_neg = [4, 8, 20, 30, 0]                 # the last session has no negative: excluded and counted as skipped
    m = impression_metrics(impression_sums(rank, auc, n_neg))
    g = lambda r: 1.0 / math.log2(1.0 + r)
    assert m["sessions"] == 4 and m["skipped"] == 1
    assert math.isclose(m["auc"], (1.0 + 0.75 + 0.5 + 0.25) / 4)
    assert math.isclose(m["mrr"], (1 + 1 / 3 + 1 / 6 + 1 / 12) / 4)           # not truncated at any cut-off
    assert math.isclose(m["ndcg5"], (g(1) + g(3)) / 4)                          # rank 6 is past the cut-off of 5
    assert math.isclose(m["ndcg10"], (g(1) + g(3) + g(6)) / 4)                  # rank 12 is past 10
    # sums add up across batches / ranks
    a = impression_sums(rank[:2], auc[:2], n_neg[:2])
    b = impression_sums(rank[2:], auc[2:], n_neg[2:])
    assert np.allclose(a + b, impression_sums(rank, auc, n_neg))


def test_impression_metrics_without_any_negative():
    from tcar_b200.util import impression_metrics, impression_sums
    m = impression_metrics(impression_sums([1, 1], [float("nan")] * 2, [0, 0]))
    assert m["sessions"] == 0 and m["skipped"] == 2 and math.isnan(m["auc"]) and math.isnan(m["mrr"])


def test_impression_eval_flag():
    from tcar_b200.main import build_parser
    assert build_parser().parse_args([]).impression_eval is False
    assert build_parser().parse_args(["--impression_eval"]).impression_eval is True
