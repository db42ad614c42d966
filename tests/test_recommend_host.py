"""Host side of the top-K recommendation (no GPU): the CLI flags, the HR / MRR / nDCG@K definitions, the output lines."""
import math

import numpy as np
import pytest


def test_recommend_flags():
    from tcar_b200.main import build_parser
    a = build_parser().parse_args([])
    assert a.recommend_k is None and a.recommend_exclude_clicked is False
    a = build_parser().parse_args(["--recommend_k", "100", "--recommend_exclude_clicked"])
    assert a.recommend_k == 100 and a.recommend_exclude_clicked is True
    assert build_parser().parse_args(["--recommend_k", "256"]).recommend_k == 256
    for bad in ("0", "257", "x"):
        with pytest.raises(SystemExit):
            build_parser().parse_args(["--recommend_k", bad])


def test_label_positions():
    from tcar_b200.util import label_positions
    ids = np.array([[5, 3, 9], [1, 2, 4], [7, -1, -1]], dtype=np.int32)
    assert label_positions(ids, [9, 8, 7]).tolist() == [3, 0, 1]


def test_topk_metrics_hand_worked():
    from tcar_b200.util import topk_metrics, topk_sums
    rank = [1, 3, 0, 20, 0]                         # 0 = the label is not in the returned list
    m = topk_metrics(topk_sums(rank))
    g = lambda r: 1.0 / math.log2(1.0 + r)
    assert m["sessions"] == 5
    assert math.isclose(m["hr"], 3 / 5)
    assert math.isclose(m["mrr"], (1 + 1 / 3 + 1 / 20) / 5)
    assert math.isclose(m["ndcg"], (g(1) + g(3) + g(20)) / 5)
    # sums add up across batches / ranks
    assert np.allclose(topk_sums(rank[:2]) + topk_sums(rank[2:]), topk_sums(rank))


def test_topk_metrics_agree_with_the_reference_cutoff_metrics():
    """With rank = 1 + #(scores above the label) and no ties, HR / MRR / nDCG@20 are util.cau_metrics' Recall / MRR /
    nDCG@20 (util.py:8-18)."""
    from tcar_b200.util import cau_metrics, label_positions, topk_metrics, topk_sums
    rs = np.random.RandomState(0)
    S = rs.randn(64, 300)
    labels = rs.randint(0, 300, 64)
    top = np.argsort(-S, axis=1)[:, :20]
    m = topk_metrics(topk_sums(label_positions(top, labels)))
    recall, mrr, ndcg = cau_metrics(S, labels)
    assert math.isclose(m["hr"], np.mean(recall)) and math.isclose(m["mrr"], np.mean(mrr))
    assert math.isclose(m["ndcg"], np.mean(ndcg))


def test_topk_metrics_of_nothing():
    from tcar_b200.util import topk_metrics, topk_sums
    m = topk_metrics(topk_sums([]))
    assert m["sessions"] == 0 and math.isnan(m["hr"])


def test_recommend_line_maps_to_original_article_ids():
    from tcar_b200.util import recommend_line
    reverse = {0: "art-17", 1: 90210, 2: "n33"}
    line = recommend_line("s_5", np.array([2, 0, -1], np.int32), np.array([1.5, -0.25, -np.inf], np.float32), reverse)
    assert line == "s_5 n33:1.5 art-17:-0.25\n"
    # nine significant digits read back the fp32 score exactly
    s = np.float32(0.1234567891)
    pair = recommend_line(7, np.array([1]), np.array([s]), reverse).split()[1]
    assert pair.split(":")[0] == "90210" and np.float32(float(pair.split(":")[1])) == s
