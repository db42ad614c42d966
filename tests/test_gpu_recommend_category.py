"""Top-K recommendation with at most C items per category and per-session allowed categories (set_item_categories /
recommend(max_per_category=..., categories=...) / tcar_recommend_category / recommend_split with
recommend_max_per_category): the result against an fp64 greedy reference, against recommend() where the two must
agree bit for bit, exact ties across categories, host checks, the rebuild of iext_cat after training, and main.py end
to end."""
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from recommend_ref import GLOBO_N, check_topk, excluded_sets, make_lists, oracle_scores, own_order_ok  # noqa: E402
from test_gpu_parity import batch_for, build  # noqa: E402


def make_codes(rs, N, G, K):
    """N codes in [0, G) with the last category cut down to K // 2 + 1 items (fewer than K: padding)."""
    cat = rs.randint(0, G - 1, N).astype(np.int64)
    cat[rs.choice(N, K // 2 + 1, replace=False)] = G - 1
    return cat


def make_allowed(rs, B, G):
    """Per-session allowed sets of five kinds: every category / one / ~10 % with duplicates / the small last category /
    none.  Returns (off, codes, the sets)."""
    sets, lists = [], []
    for b in range(B):
        kind = b % 5
        if kind == 0:
            lst = list(range(G))
        elif kind == 1:
            lst = [int(rs.randint(0, G - 1))]
        elif kind == 2:
            lst = rs.choice(G, max(1, G // 10), replace=False).tolist()
            lst = lst + lst[:2]
        elif kind == 3:
            lst = [G - 1]
        else:
            lst = []
        sets.append(set(lst))
        lists.append(lst)
    off = np.cumsum([0] + [len(x) for x in lists]).astype(np.int32)
    codes = np.array([c for x in lists for c in x], np.int32)
    return off, codes, sets


@pytest.mark.parametrize("B,N,G,K,C,kind", [(20, 30000, 5, 1, 1, "plain"), (40, 30000, 17, 20, 2, "clicked"),
                                            (30, 30000, 300, 256, 1, "dup"), (25, 30000, 17, 256, 2, "clicked"),
                                            (15, 30000, 264, 20, 20, "plain"),
                                            (24, GLOBO_N, 461, 20, 2, "clicked"), (10, GLOBO_N, 461, 256, 256, "dup"),
                                            (10, GLOBO_N, 17, 100, 1, "plain")])
def test_category_matches_fp64_reference(B, N, G, K, C, kind):
    T = 3
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=B + K + G)
    rs = np.random.RandomState(G + K)
    cat = make_codes(rs, N, G, K)
    model.set_item_categories(cat)
    a_off, a_codes, sets = make_allowed(rs, B, G)
    off = lst = None
    clicked = kind == "clicked"
    if kind == "dup":
        off, lst = make_lists(rs, N, rs.randint(0, 300, B).tolist(), dup=True)
    ex = excluded_sets(B, off, lst, batch["seq"].numpy() if clicked else None)
    S = oracle_scores(model, content, mwdhm, batch)
    for allowed, sets_ in (((a_off, a_codes), sets), (None, [None] * B)):
        kw = dict(exclude_off=off, exclude_ids=lst, exclude_clicked=clicked, max_per_category=C, categories=allowed)
        ids, sc = [x.clone() for x in model.recommend(bt, K, **kw)]
        ids2, sc2 = model.recommend(bt, K, **kw)
        torch.cuda.synchronize()
        assert torch.equal(ids, ids2) and torch.equal(sc, sc2), "a second run must be bit-identical"
        ids_h, sc_h = ids.cpu().numpy(), sc.cpu().numpy()
        margin = check_topk(ids_h, sc_h, S, K, ex, C, cat, sets_)
        if K <= 100:
            assert margin.mean() > 0.5, "fixture must be mostly margin-checked"
        if allowed is not None:
            assert all((ids_h[b] == -1).all() for b in range(B) if b % 5 == 4), "no category allowed: all -1"
            assert K == 1 or all((ids_h[b] == -1).any() for b in range(B) if b % 5 == 3), "fewer than K: padded"
            assert (model.rec_rescored[:B].cpu().numpy()[4::5] == 0).all(), "nothing allowed re-scores nothing"


@pytest.mark.parametrize("N,G", [(30000, 17), (GLOBO_N, 461)])
def test_uncapped_all_categories_equals_recommend(N, G):
    """C >= K with every category allowed is recommend() itself: ids and scores with torch.equal."""
    B, T = 64, 4
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=5)
    rs = np.random.RandomState(3)
    model.set_item_categories(rs.randint(0, G, N))
    off, lst = make_lists(rs, N, rs.randint(0, 200, B).tolist(), dup=True)
    every = (np.arange(B + 1, dtype=np.int32) * G, np.tile(np.arange(G, dtype=np.int32), B))
    for K in (20, 256):
        for kw in ({}, dict(exclude_off=off, exclude_ids=lst, exclude_clicked=True)):
            a = [x.clone() for x in model.recommend(bt, K, **kw)]
            for extra in (dict(max_per_category=K), dict(max_per_category=10 ** 9, categories=every),
                          dict(categories=every)):
                c = model.recommend(bt, K, **kw, **extra)
                torch.cuda.synchronize()
                assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1]), (K, kw.keys(), extra.keys())


def test_allowed_set_equals_complement_exclusion_list():
    """Without a cap, an allowed set gives recommend() with the complement as its exclusion list, bit for bit."""
    from tcar_b200 import _native as nv
    N, B, T, K, G = 1500, 48, 3, 50, 40
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=23)
    rs = np.random.RandomState(6)
    cat = rs.randint(0, G, N)
    model.set_item_categories(cat)
    sets = [rs.choice(G, 30, replace=False) for _ in range(B)]
    a_off = np.cumsum([0] + [len(s) for s in sets]).astype(np.int32)
    a_codes = np.concatenate(sets).astype(np.int32)
    out = [np.flatnonzero(~np.isin(cat, s)) for s in sets]
    assert max(len(o) for o in out) + T <= nv.RECOMMEND_MAXX
    off = np.cumsum([0] + [len(o) for o in out]).astype(np.int32)
    lst = np.concatenate(out).astype(np.int32)
    for clicked in (False, True):
        a = [x.clone() for x in model.recommend(bt, K, exclude_clicked=clicked, categories=(a_off, a_codes))]
        b_ = model.recommend(bt, K, off, lst, exclude_clicked=clicked)
        torch.cuda.synchronize()
        assert torch.equal(a[0], b_[0]) and torch.equal(a[1], b_[1]), clicked
    assert (a[0] >= 0).all()


def test_identical_rows_in_different_categories():
    """Copies of one row score bit for bit the same: with C = 1 the list holds the lowest id of the row's own category
    and every copy in another category, in id order; without a cap every copy, in id order."""
    from tcar_b200.params import ParamStore
    N, B, T, G = 20000, 8, 2, 50
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=31)
    top = int(model.recommend(bt, 1)[0][0, 0])
    rs = np.random.RandomState(8)
    cat = rs.randint(0, G, N)
    same = [int(x) for x in rs.choice(np.flatnonzero((cat == cat[top]) & (np.arange(N) != top)), 2, replace=False)]
    others = [int(x) for x in rs.choice(np.flatnonzero(cat != cat[top]), 6, replace=False)]
    cat[others[3:]] = cat[others[0]]                       # three copies in one other category, three in their own
    p = model.ps.export()
    cont, mw = content.copy(), mwdhm.copy()
    for d in same + others:
        p["item"][d + 1], cont[d + 1], mw[d] = p["item"][top + 1], cont[top + 1], mw[top]
    model.ps = ParamStore(N, cont, mw, model.dev)
    model.ps.load(p)
    model.set_item_categories(cat)
    bt, _ = batch_for(model, N, B, T, 0, mw, seed=31)
    copies = sorted([top] + same + others)
    ids, sc = model.recommend(bt, 20, max_per_category=1)
    ids_u, sc_u = model.recommend(bt, 20, max_per_category=20)
    torch.cuda.synchronize()
    ids, sc, ids_u, sc_u = (x.cpu().numpy() for x in (ids, sc, ids_u, sc_u))
    own_order_ok(ids, sc)
    assert ids_u[0, :len(copies)].tolist() == copies and len(set(sc_u[0, :len(copies)].tolist())) == 1
    first = {}
    for j in copies:
        first.setdefault(int(cat[j]), j)
    want = sorted(first.values())
    assert ids[0, :len(want)].tolist() == want and (sc[0, :len(want)] == sc_u[0, 0]).all()


def test_category_host_checks_launch_nothing():
    from tcar_b200 import _native as nv
    N, B, T, G = 500, 4, 2, 7
    model, _, mwdhm, _ = build(N)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=1)
    before = nv.LAUNCHES["count"]
    with pytest.raises(ValueError, match="set_item_categories"):
        model.recommend(bt, 5, max_per_category=2)
    with pytest.raises(ValueError, match="set_item_categories"):
        model.recommend(bt, 5, categories=(np.zeros(B + 1, int), np.zeros(0, int)))
    for codes, G_, what in [(np.zeros(N - 1, int), None, f"N = {N}"), (np.full(N, -1), None, "item 0"),
                            (np.arange(N) % 9, G, "item 7: category 7 outside"), (np.zeros(N), None, "integers"),
                            (np.arange(N) % 2, 1025, "TCAR_RECOMMEND_MAXG")]:
        with pytest.raises(ValueError, match=what):
            model.set_item_categories(codes, G_)
    assert getattr(model, "_iext_cat", None) is None
    model.set_item_categories(np.arange(N) % G)
    good = (np.array([0, 1, 1, 3, 3]), np.array([2, 0, 6], np.int32))
    for kw, what in [(dict(max_per_category=0), "max_per_category"), (dict(max_per_category=True), "max_per_category"),
                     (dict(max_per_category=2.0), "max_per_category"),
                     (dict(categories=np.zeros(5, int)), "pair"),
                     (dict(categories=(np.array([0, 1, 1, 3]), good[1])), "B \\+ 1 = 5"),
                     (dict(categories=(good[0], np.array([2, 0, 7]))), "session 2: category 7 outside \\[0, 7\\)"),
                     (dict(categories=good, window=(np.zeros(B, int), np.ones(B, int))), "window"),
                     (dict(max_per_category=2, exclude_off=np.array([0, 0, 0, 0, 1]), exclude_ids=np.array([N])),
                      "outside")]:
        if "window" in kw:
            model.set_item_times(np.arange(N))
        with pytest.raises(ValueError, match=what):
            model.recommend(bt, 5, **kw)
    assert nv.LAUNCHES["count"] == before, "validation happens before any launch"
    # the C entry point refuses bad limits and missing inputs
    p = nv.ptr
    buf = torch.zeros(model._cat_n_pad * 4, device=model.dev)
    ws = torch.zeros(int(nv.lib().tcar_recommend_category_ws_bytes(B)), device=model.dev, dtype=torch.uint8)
    base = [p(buf)] * 7 + [None, None, None, T, B, model._cat_n_pad, 5, p(buf), p(buf), p(buf), G, None, None, 2,
                           p(ws), p(buf), p(buf), None, nv.stream_ptr()]
    for at, val in ((17, 0), (17, 1025), (20, 0), (14, None), (16, None), (21, None), (13, 257), (12, 100)):
        a = list(base)
        a[at] = val
        assert nv.lib().tcar_recommend_category(*a) == -1, (at, val)
    torch.cuda.synchronize()


def test_iext_cat_rebuilt_after_train_step():
    """A train step changes the item table: the category-ordered copy follows, so the result equals that of a model
    restored from the same state."""
    N, B, T, K, G = 3000, 32, 4, 20, 23
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    cat = np.random.RandomState(2).randint(0, G, N)
    model.set_item_categories(cat)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=4)
    before = [x.clone() for x in model.recommend(bt, K, max_per_category=2, exclude_clicked=True)]
    tb, _ = batch_for(model, N, 64, 5, 20, mwdhm, seed=9)
    for _ in range(3):
        model.train_step(tb)
    after = [x.clone() for x in model.recommend(bt, K, max_per_category=2, exclude_clicked=True)]
    assert torch.equal(model._iext_cat[:model._cat_n], model.ps.iext[model._cat_src]), "the copy follows the table"
    assert not model._iext_cat[model._cat_n:].any()
    fresh, _, _, _ = build(N, emb_scale=20.0)
    fresh.ps.load_state_dict(model.ps.state_dict())
    fresh.set_item_categories(cat)
    bt2, _ = batch_for(fresh, N, B, T, 0, mwdhm, seed=4)
    want = fresh.recommend(bt2, K, max_per_category=2, exclude_clicked=True)
    torch.cuda.synchronize()
    assert torch.equal(after[0], want[0]) and torch.equal(after[1], want[1])
    assert not torch.equal(before[1], after[1]), "training must have moved the scores"


def test_recommend_split_max_per_category_end_to_end(tmp_path, monkeypatch):
    """main.py --recommend_k 20 --recommend_max_per_category 2 on a synthetic split: every written list holds at most
    two articles of one category, and the printed ILD / unexpectedness are those of the written lists."""
    from tcar_b200 import main as tmain, synth
    from tcar_b200.util import list_ild, list_unexp
    N, n_test = 1500, 150
    monkeypatch.chdir(tmp_path)
    root = str(tmp_path) + "/synth/TCAR-mid/Normal/"
    synth.write_dataset(root, N=N, n_train=700, n_test=n_test, fold=0)
    args = tmain.build_parser().parse_args(["--datapath", str(tmp_path) + "/", "--dataset", "synth/TCAR-mid/",
                                            "--foldnum", "0", "--epoch", "1", "--batch_size", "64",
                                            "--recommend_k", "20", "--recommend_max_per_category", "2",
                                            "--recommend_exclude_clicked"])
    model = tmain.main(args)
    got = model.last_recommend_metrics
    load = lambda name: pickle.load(open(root + name, "rb"))
    art_cat, item_dict, sdict = load("articles_category.pkl"), load("item_dict_0.txt"), load("session_dict_test_0.pkl")
    rev = {v: k for k, v in item_dict.items()}
    lines = open(tmp_path / "saved" / "recommend_0.txt").read().splitlines()
    assert len(lines) == n_test == got["sessions"]
    ild = unexp = 0.0
    for line in lines:
        key, *pairs = line.split()
        arts = [a.rsplit(":", 1)[0] for a in pairs]
        cats = [art_cat[a] for a in arts]
        assert len(arts) == 20 and max(cats.count(c) for c in cats) <= 2
        ild += list_ild(cats)
        unexp += list_unexp(cats, [art_cat[rev[i]] for i in sdict[int(key)][:-1]])
    np.testing.assert_allclose([got["ild"], got["unexp"]], [ild / n_test, unexp / n_test], rtol=1e-12)


def test_few_categories_small_cap_scan_each_category_to_its_own_bound():
    """|M| <= K' (17 categories, C = 1, K = 20, clicks excluded): no global threshold exists, and each category is
    scanned only down to its own (C + x_b)-th chunk maximum - 2 eps_b, not the whole catalog."""
    N, B, T, G, K = 30000, 64, 3, 17, 20
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=41)
    cat = np.random.RandomState(7).randint(0, G, N)
    model.set_item_categories(cat)
    ex = excluded_sets(B, None, None, batch["seq"].numpy())
    S = oracle_scores(model, content, mwdhm, batch)
    for C in (1, 2):
        ids, sc = [x.clone() for x in model.recommend(bt, K, exclude_clicked=True, max_per_category=C)]
        torch.cuda.synchronize()
        margin = check_topk(ids.cpu().numpy(), sc.cpu().numpy(), S, K, ex, C, cat)
        assert margin.mean() > 0.5
        assert (ids.cpu().numpy()[:, G * C:] == -1).all() and (ids.cpu().numpy()[:, :G * C] >= 0).all()
        assert model.rec_rescored[:B].float().mean().item() < N / 10, "each category to its own bound, not all of it"


def _skewed_model(N, G, big_share, seed):
    """A catalog whose category 0 holds big_share of the items; the rest split evenly."""
    rs = np.random.RandomState(seed)
    cat = rs.randint(1, G, N)
    cat[rs.rand(N) < big_share] = 0
    return cat


@pytest.mark.parametrize("N", [60000, GLOBO_N])
def test_capped_select_counts_every_chunk_when_the_list_is_not_enough(N):
    """One category holds 99.7 % of the items: the 4 096 best chunks give fewer than K' capped entries, so the select
    counts over every allowed chunk (its fallback) -- the result still equals the reference."""
    B, T, G, K, C = 16, 2, 40, 30, 1
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=43)
    cat = _skewed_model(N, G, 0.997, 5)
    model.set_item_categories(cat, G)
    ids, sc = model.recommend(bt, K, max_per_category=C)
    torch.cuda.synchronize()
    S = oracle_scores(model, content, mwdhm, batch)
    check_topk(ids.cpu().numpy(), sc.cpu().numpy(), S, K, [set() for _ in range(B)], C, cat)


def test_capped_select_with_more_tied_chunks_than_its_list():
    """Identical rows in more than 4 096 chunks tie at the top: the list of the capped select overflows and it counts
    over every allowed chunk; ties resolve to the lower id in every category."""
    from tcar_b200.params import ParamStore
    N, B, T, G, K, C = 60000, 8, 2, 461, 20, 2
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=47)
    top = int(model.recommend(bt, 1)[0][0, 0])
    rs = np.random.RandomState(9)
    cat = rs.randint(0, G, N)
    # the batch's clicks and labels keep their rows, so the sessions' queries do not move and session 0's best row is
    # the tied one
    keep = np.union1d(batch["seq"].numpy().reshape(-1) - 1, batch["label"].numpy() - 1)
    copies = rs.choice(np.setdiff1d(np.arange(N), np.append(keep, top)), 40000, replace=False)
    p = model.ps.export()
    cont, mw = content.copy(), mwdhm.copy()
    p["item"][copies + 1] = p["item"][top + 1].clone()
    cont[copies + 1], mw[copies] = cont[top + 1], mw[top]
    model.ps = ParamStore(N, cont, mw, model.dev)
    model.ps.load(p)
    model.set_item_categories(cat, G)
    bt, batch = batch_for(model, N, B, T, 0, mw, seed=47)
    ids, sc = model.recommend(bt, K, max_per_category=C)
    torch.cuda.synchronize()
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    own_order_ok(ids, sc)
    tied = np.union1d(copies, [top])
    want, used = [], {}
    for j in tied:                                           # session 0: its top is the tied row
        if used.get(cat[j], 0) < C:
            used[cat[j]] = used.get(cat[j], 0) + 1
            want.append(int(j))
            if len(want) == K:
                break
    assert ids[0].tolist() == want and (sc[0] == sc[0, 0]).all()
    S = oracle_scores(model, cont, mw, batch)
    check_topk(ids, sc, S, K, [set() for _ in range(B)], C, cat)
