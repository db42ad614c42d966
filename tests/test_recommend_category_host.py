"""Host side of top-K recommendation by category (no GPU): the category-ordered layout, an fp64 greedy reference of the
capped, filtered top-K, the ValueErrors of set_item_categories / recommend(max_per_category=..., categories=...), the
--recommend_max_per_category flag, the split's category codes and the ILD / unexpectedness helpers."""
import types

import numpy as np
import pytest

from recommend_ref import topk_ref


def check_layout(codes, G):
    from tcar_b200.util import category_layout, pad_sources
    codes = np.asarray(codes)
    N = len(codes)
    perm, off, n2 = category_layout(codes, G)
    assert perm.dtype == np.int32 and off.dtype == np.int32 and off.shape == (G + 1,)
    assert n2 == len(perm) == 8 * off[G] and n2 % 8 == 0 and n2 <= N + 7 * G
    real = perm[perm >= 0]
    assert sorted(real.tolist()) == list(range(N)), "every item exactly once"
    src = pad_sources(perm)
    for g in range(G):
        lo, hi = 8 * off[g], 8 * off[g + 1]
        items = np.flatnonzero(codes == g)
        assert off[g + 1] - off[g] == (len(items) + 7) // 8, "whole chunks, empty categories empty"
        assert perm[lo:lo + len(items)].tolist() == items.tolist(), "sorted by (code, id)"
        assert (perm[lo + len(items):hi] == -1).all()
        if len(items):
            assert (src[lo + len(items):hi] == items[-1]).all(), "a pad repeats its category's last item"
    assert (src[perm >= 0] == perm[perm >= 0]).all()
    return perm, off


def test_layout_random_and_edge_cases():
    rs = np.random.RandomState(0)
    check_layout(rs.randint(0, 17, 1000), 17)
    check_layout(rs.randint(0, 461, 5000), 461)
    perm, off = check_layout(np.zeros(13, int), 1)                      # G = 1
    assert off.tolist() == [0, 2] and perm[13:].tolist() == [-1, -1, -1]
    perm, off = check_layout(np.array([3, 3, 0, 3]), 5)                 # empty categories 1, 2, 4
    assert off.tolist() == [0, 1, 1, 1, 2, 2]
    assert perm.tolist() == [2] + [-1] * 7 + [0, 1, 3] + [-1] * 5
    codes = np.arange(2048) % 1024                                      # G = 1024: two items each
    perm, off = check_layout(codes, 1024)
    assert len(perm) == 8 * 1024
    check_layout(np.full(16, 2), 3)                                     # exactly whole chunks: no pad
    check_layout(np.zeros(0, int), 4)


def capped_topk(S, K, C, cat, allowed=None, excluded=()):
    """fp64 greedy reference of one row: by (score desc, id asc), drop an item with C items of its category before it
    or outside the allowed categories or excluded; the first K."""
    order = np.lexsort((np.arange(len(S)), -S))
    out, used = [], {}
    for j in order:
        if j in excluded or (allowed is not None and cat[j] not in allowed):
            continue
        if used.get(cat[j], 0) < C:
            used[cat[j]] = used.get(cat[j], 0) + 1
            out.append(int(j))
            if len(out) == K:
                break
    return out


def test_capped_reference_properties():
    """Capping is decomposable: the capped top-K of A u B is the capped top-K of the two capped lists' union (what the
    per-CTA lists and their final merge rely on), and C >= K is no cap.  recommend_ref.topk_ref agrees with this
    brute force."""
    rs = np.random.RandomState(1)
    N, G = 400, 9
    cat = rs.randint(0, G, N)
    for trial in range(20):
        S = np.round(rs.randn(N), 1)                                    # many exact ties: id order decides
        K, C = int(rs.randint(1, 40)), int(rs.randint(1, 6))
        allowed = set(rs.choice(G, 5, replace=False).tolist()) if trial % 2 else None
        ex = set(rs.choice(N, 30).tolist())
        want = capped_topk(S, K, C, cat, allowed, ex)
        split = rs.randint(0, 4, N)
        parts = [capped_topk(np.where(split == s, S, -np.inf), K, C, cat, allowed, ex) for s in range(4)]
        parts = [[j for j in p if split[j] == s] for s, p in enumerate(parts)]
        union = np.full(N, -np.inf)
        for p in parts:
            union[p] = S[p]
        assert capped_topk(union, K, C, cat, allowed, ex) == [j for j in want], trial
        assert capped_topk(S, K, K, cat) == capped_topk(S, K, 10 ** 9, cat)
        assert all(np.bincount(cat[want], minlength=G).max(initial=0) <= C for _ in [0])
        # the fp64 reference of the GPU tests: row by row the brute force above, and without a cap or categories the
        # same ids, scores and margins as with C = K and one category
        rows = np.stack([S, np.round(rs.randn(N), 1), np.round(rs.randn(N), 3)])
        r_ex = [ex, set(), set(rs.choice(N, 10).tolist())]
        r_allowed = [allowed, None, set(rs.choice(G, 3, replace=False).tolist())]
        r_ids = topk_ref(rows, K, r_ex, C, cat, r_allowed)[0]
        for row, r_row in zip(range(3), r_ids):
            assert r_row[r_row >= 0].tolist() == capped_topk(rows[row], K, C, cat, r_allowed[row], r_ex[row]), trial
        plain = topk_ref(rows, K, r_ex)
        one_cat = topk_ref(rows, K, r_ex, K, np.zeros(N, np.int64), [None] * 3)
        assert all(np.array_equal(x, y) for x, y in zip(plain, one_cat)), trial


def test_item_category_checks():
    from tcar_b200.util import check_item_categories
    c, G = check_item_categories(np.array([0, 3, 1], np.uint8), 3)
    assert c.dtype == np.int32 and G == 4
    assert check_item_categories([0, 0], 2, 1024)[1] == 1024
    for codes, G, what in [([0, 1], None, "N = 3"), ([0, -1, 0], None, "item 1: category -1"),
                           ([0, 5, 0], 5, "item 1: category 5 outside \\[0, 5\\)"), ([0.0, 1, 2], None, "integers"),
                           ([0, 1, 2], 1025, "TCAR_RECOMMEND_MAXG = 1024"), ([0, 1, 2], 0, "MAXG"),
                           ([0, 1, 2], True, "MAXG"), ([0, 1, 1024], None, "MAXG")]:
        with pytest.raises(ValueError, match=what):
            check_item_categories(np.asarray(codes), 3, G)


def test_model_checks_raise_before_anything_is_uploaded():
    from tcar_b200.model_combine import Seq2SeqAttNN
    m = Seq2SeqAttNN.__new__(Seq2SeqAttNN)
    m.N = 5
    for codes, what in [([0, 0, 0, 0, 2000], "MAXG"), ([0, 0, 0, 0, -1], "item 4"), ([0, 0], "N = 5")]:
        with pytest.raises(ValueError, match=what):
            m.set_item_categories(codes)
    assert getattr(m, "_iext_cat", None) is None
    bt = types.SimpleNamespace(B=2, T=3)
    for kw in (dict(max_per_category=2), dict(categories=([0, 0, 0], []))):
        with pytest.raises(ValueError, match="set_item_categories"):
            m.recommend(bt, 5, **kw)
    m._iext_cat, m._cat_G, m._item_time = object(), 4, object()        # as if set: the argument checks come next
    for kw, what in [(dict(max_per_category=0), "max_per_category"), (dict(max_per_category=False), "integer"),
                     (dict(max_per_category=1.5), "integer"), (dict(categories=[0, 0, 0]), "pair"),
                     (dict(categories=([0, 1], [2])), "B \\+ 1 = 3"),
                     (dict(categories=([0, 2, 1], [0])), "session 1: categories off decreases"),
                     (dict(categories=([0, 1, 2], [0, 4])), "session 1: category 4 outside \\[0, 4\\)"),
                     (dict(categories=([0, 1, 2], [0.0, 1.0])), "integers"),
                     (dict(max_per_category=2, window=([0, 0], [1, 1])), "window cannot be combined")]:
        with pytest.raises(ValueError, match=what):
            m.recommend(bt, 5, **kw)


def test_max_per_category_flag():
    from tcar_b200.main import build_parser
    a = build_parser().parse_args(["--recommend_k", "20", "--recommend_max_per_category", "2",
                                   "--recommend_exclude_clicked"])
    assert a.recommend_max_per_category == 2 and a.recommend_exclude_clicked
    assert build_parser().parse_args([]).recommend_max_per_category is None
    for argv in (["--recommend_k", "20", "--recommend_max_per_category", "0"],
                 ["--recommend_k", "20", "--recommend_max_per_category", "x"],
                 ["--recommend_max_per_category", "2"],
                 ["--recommend_k", "20", "--recommend_max_per_category", "2", "--recommend_max_age_h", "24"]):
        with pytest.raises(SystemExit):
            build_parser().parse_args(argv)


def test_split_codes_share_one_unknown_code():
    from tcar_b200.model_combine import Seq2SeqAttNN
    m = Seq2SeqAttNN.__new__(Seq2SeqAttNN)
    m.N = 6
    m.reverse_item = {i: "a%d" % i for i in range(6)}
    m.category_id = {"a0": "sport", "a1": "news", "a2": "sport", "a4": "news"}      # a3, a5: no category
    assert m._split_category_codes().tolist() == [0, 1, 0, 2, 1, 2]
    m.category_id, m.reverse_item = [7, 7, 3, 9, 3, 7], list(range(6))             # a plain array of codes
    assert m._split_category_codes().tolist() == [0, 0, 1, 2, 1, 0]


def test_ild_and_unexpectedness():
    from tcar_b200.util import diversity_sums, list_ild, list_unexp
    assert list_ild([1, 1, 2]) == pytest.approx(4 / 6)
    assert list_ild([5]) == 0.0 and list_ild([]) == 0.0
    assert list_ild([1, 2, 3]) == 1.0
    assert list_unexp([1, 2], [1, 1, 3]) == pytest.approx(4 / 6)
    assert list_unexp([], [1]) == 0.0
    cat = np.array([0, 0, 1, 2, 1])
    ids = np.array([[0, 2, -1], [3, 4, 1], [-1, -1, 2]])
    got = diversity_sums(ids, [[1], [2, 3], [0]], cat)
    want = [list_ild([0, 1]) + list_ild([2, 1, 0]), list_unexp([0, 1], [0]) + list_unexp([2, 1, 0], [1, 2]), 2]
    np.testing.assert_allclose(got, want)                               # a list of one item is left out, as in test()
