"""Top-K recommendation (tcar_recommend / Seq2SeqAttNN.recommend / recommend_split) against an fp64 reference built on
the oracle's forward(), against the full-catalog evaluation it must agree with bit for bit, and against itself with and
without exclusions.

Reference: the oracle's softmax_input (model_combine.py:138) with the excluded ids set to -inf, ordered by (score desc,
id asc) and cut to K."""
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import tcar_oracle as O  # noqa: E402
from test_gpu_parity import batch_for, build, oracle_inputs  # noqa: E402

GLOBO_N = 364047


def oracle_scores(model, content, mwdhm, batch):
    params, c64, m64 = oracle_inputs(model, content, mwdhm)
    with torch.no_grad():
        return O.forward(params, c64, m64, batch)["softmax_input"].numpy()


def recommend_ref(S, K, excluded):
    """fp64 reference: per row the K best eligible items by (score desc, id asc), padded with -1 / -inf, and whether
    the first K + 1 eligible scores are separated by more than 2e-5 |score| (the margin_ok rule)."""
    B, N = S.shape
    ids = np.full((B, K), -1, np.int64)
    sc = np.full((B, K), -np.inf)
    margin = np.zeros(B, bool)
    for b in range(B):
        s = S[b].copy()
        ex = np.array(sorted(excluded[b]), np.int64)
        s[ex] = -np.inf
        order = np.lexsort((np.arange(N), -s))
        order = order[np.isfinite(s[order])]
        n = min(K, len(order))
        ids[b, :n], sc[b, :n] = order[:n], s[order[:n]]
        head = s[order[:K + 1]]
        margin[b] = len(head) < 2 or bool((np.abs(np.diff(head)) > 2e-5 * np.abs(head).max()).all())
    return ids, sc, margin


def own_order_ok(ids, sc):
    """Every row is ordered exactly by (score desc, id asc) of its own fp32 scores, padding last."""
    for i_row, s_row in zip(ids, sc):
        n = int((i_row >= 0).sum())
        assert (i_row[n:] == -1).all() and np.isneginf(s_row[n:]).all()
        i, s = i_row[:n].astype(np.int64), s_row[:n].astype(np.float64)
        assert (np.lexsort((i, -s)) == np.arange(n)).all()
        assert len(set(i.tolist())) == n


def make_lists(rs, N, lens, dup=False):
    off = np.zeros(len(lens) + 1, dtype=np.int32)
    off[1:] = np.cumsum(lens)
    ids = rs.randint(0, N, int(off[-1])).astype(np.int32)
    if dup:
        for b, L in enumerate(lens):
            if L > 2:
                ids[off[b] + L - 1] = ids[off[b]]
                ids[off[b] + 1] = ids[off[b]]
    return off, ids


def excluded_sets(B, off, ids, seq=None):
    ex = [set() for _ in range(B)]
    if off is not None:
        for b in range(B):
            ex[b].update(ids[off[b]:off[b + 1]].tolist())
    if seq is not None:
        for b in range(B):
            ex[b].update((seq[b] - 1).tolist())
    return ex


def check_against_reference(ids, sc, S, K, excluded):
    r_ids, r_sc, margin = recommend_ref(S, K, excluded)
    own_order_ok(ids, sc)
    valid = r_ids >= 0
    assert ((ids >= 0) == valid).all(), "padding where the reference has no eligible item"
    np.testing.assert_allclose(sc[valid], r_sc[valid], rtol=1e-4, atol=1e-5)
    assert (ids[margin] == r_ids[margin]).all(), "ids exact on margin-checked rows"
    # every row: the returned items are eligible and are as good as the reference's, position by position
    for b in range(len(ids)):
        got = ids[b][ids[b] >= 0]
        assert not (set(got.tolist()) & excluded[b])
        np.testing.assert_allclose(S[b, got], r_sc[b, :len(got)], rtol=1e-4, atol=1e-5)
    return margin


@pytest.mark.parametrize("B,N,K,T,kind", [(1, 300, 1, 1, "plain"), (7, 2000, 100, 3, "dup"),
                                          (512, 9000, 256, 20, "clicked"), (64, 70000, 256, 2, "maxx"),
                                          (5, 300, 256, 4, "small")])
def test_recommend_matches_fp64_reference(B, N, K, T, kind):
    from tcar_b200 import _native as nv
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=B + K)
    rs = np.random.RandomState(K)
    off = lst = None
    clicked = kind in ("clicked", "small")
    if kind == "dup":
        off, lst = make_lists(rs, N, [0, 1, 5, 37, 100, 3, 250], dup=True)
    elif kind == "maxx":
        off, lst = make_lists(rs, N, [nv.RECOMMEND_MAXX] + rs.randint(0, nv.RECOMMEND_MAXX + 1, B - 1).tolist())
    elif kind == "small":
        off, lst = make_lists(rs, N, [40, 0, 100, 7, 60])
    kw = dict(exclude_off=off, exclude_ids=lst, exclude_clicked=clicked)
    ids, sc = [x.clone() for x in model.recommend(bt, K, **kw)]
    ids2, sc2 = model.recommend(bt, K, **kw)
    torch.cuda.synchronize()
    assert torch.equal(ids, ids2) and torch.equal(sc, sc2), "a second run must be bit-identical"
    S = oracle_scores(model, content, mwdhm, batch)
    ex = excluded_sets(B, off, lst, batch["seq"].numpy() if clicked else None)
    margin = check_against_reference(ids.cpu().numpy(), sc.cpu().numpy(), S, K, ex)
    if K <= 100:
        assert margin.mean() > 0.5, "fixture must be mostly margin-checked"
    if kind == "small":
        assert (ids.cpu().numpy() == -1).any(), "fewer eligible items than K: padded"


@pytest.mark.parametrize("N,B,T", [(30000, 256, 4), (GLOBO_N, 64, 20)])
def test_recommend_agrees_bit_for_bit_with_eval_step(N, B, T):
    """K <= 20 without exclusions: the prefix of eval_step's certified top-20, ids and scores, with torch.equal."""
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=N % 97)
    top, _, _ = model.eval_step(bt)
    top, top_sc = top.clone(), model.top_scores[:B].clone()
    for K in (20, 7, 1):
        ids, sc = model.recommend(bt, K)
        torch.cuda.synchronize()
        assert torch.equal(ids, top[:, :K]), K
        assert torch.equal(sc, top_sc[:, :K]), K


def test_exclusions_equal_filtering_a_longer_list():
    """recommend(K, exclusions) == recommend(K + x) without them, the excluded ids removed, cut to K -- bit for bit;
    exclude_clicked == the clicks (0-based) passed as an explicit list."""
    N, B, T, K = 20000, 96, 5, 60
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=17)
    full_ids, full_sc = [x.cpu().numpy() for x in model.recommend(bt, 256)]
    rs = np.random.RandomState(3)
    # exclusions drawn partly from each session's own top list (so that they matter), partly at random, with repeats
    lists = []
    for b in range(B):
        x = rs.randint(0, 80)
        pick = full_ids[b, rs.choice(K + x, min(x, K + x), replace=False)].tolist() + rs.randint(0, N, 5).tolist()
        lists.append(pick + pick[:3])
    lens = [len(x) for x in lists]
    assert K + max(lens) <= 256
    off = np.cumsum([0] + lens).astype(np.int32)
    lst = np.concatenate(lists).astype(np.int32)
    ids, sc = [x.cpu().numpy() for x in model.recommend(bt, K, off, lst)]
    for b in range(B):
        ex = set(lists[b])
        keep = np.array([i not in ex for i in full_ids[b]])
        want_i, want_s = full_ids[b][keep][:K], full_sc[b][keep][:K]
        assert (ids[b] == want_i).all() and (sc[b].view(np.int32) == want_s.view(np.int32)).all(), b
    # exclude_clicked == an explicit list of the clicks
    seq = batch["seq"].numpy()
    c_off = (np.arange(B + 1) * T).astype(np.int32)
    a = [x.clone() for x in model.recommend(bt, K, exclude_clicked=True)]
    b_ = model.recommend(bt, K, c_off, (seq - 1).reshape(-1).astype(np.int32))
    torch.cuda.synchronize()
    assert torch.equal(a[0], b_[0]) and torch.equal(a[1], b_[1])
    got = a[0].cpu().numpy()
    for b in range(B):
        assert not (set(got[b].tolist()) & set((seq[b] - 1).tolist()))
    # both exclusion sources together
    c = model.recommend(bt, K, off, lst, exclude_clicked=True)[0].cpu().numpy()
    for b in range(B):
        ex = set(lists[b]) | set((seq[b] - 1).tolist())
        keep = np.array([i not in ex for i in full_ids[b]])
        assert (c[b] == full_ids[b][keep][:K]).all(), b


def test_wide_bands_near_tie_clusters():
    """Clusters of near-identical rows (scores within the bf16 error of each other) put hundreds of chunks inside the
    band: the result still equals the fp64 reference and a full exact scan."""
    N, B, T, K = 40000, 32, 2, 100
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=13)
    tops = model.recommend(bt, 1)[0][:6, 0].cpu().numpy()       # a cluster at the top of sessions 0..5
    p = model.ps.export()
    rs = np.random.RandomState(1)
    cont, mw = content.copy(), mwdhm.copy()
    for src in tops:
        src = int(src)
        dst = rs.choice(N // 8, 150, replace=False) * 8 + rs.randint(0, 8, 150)
        for d_ in dst:
            p["item"][d_ + 1] = p["item"][src + 1] * (1 + 1e-4 * float(rs.randn()))
            cont[d_ + 1] = cont[src + 1] * (1 + 1e-4 * float(rs.randn()))
            mw[d_] = mw[src]
    from tcar_b200.params import ParamStore
    model.ps = ParamStore(N, cont, mw, model.dev)
    model.ps.load(p)
    bt, batch = batch_for(model, N, B, T, 0, mw, seed=13)
    ids, sc = [x.clone() for x in model.recommend(bt, K, exclude_clicked=True)]
    n_band = model.rec_rescored[:B].cpu().numpy()
    assert n_band.max() >= 1000, "fixture should open a band of hundreds of chunks"
    S = oracle_scores(model, cont, mw, batch)
    check_against_reference(ids.cpu().numpy(), sc.cpu().numpy(), S, K,
                            excluded_sets(B, None, None, batch["seq"].numpy()))
    model.cat_stats.fill_(1e4)                  # eps_b ~ 1e4 ||q||: the band is the whole catalog
    ids2, sc2 = model.recommend(bt, K, exclude_clicked=True)
    n_full = model.rec_rescored[:B].cpu().numpy()
    torch.cuda.synchronize()
    assert (n_full >= N - T).all() and (n_full > n_band).all()
    assert torch.equal(ids, ids2) and torch.equal(sc, sc2)


def test_recommend_input_checks():
    from tcar_b200 import _native as nv
    N, B, T = 500, 4, 2
    model, _, mwdhm, _ = build(N)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=1)
    good_off, good_ids = np.array([0, 2, 3, 3, 5]), np.array([1, 2, 3, 4, 5])
    before = nv.LAUNCHES["count"]
    for k in (0, nv.RECOMMEND_MAXK + 1, 2.0, True):
        with pytest.raises(ValueError, match="k must be"):
            model.recommend(bt, k)
    long = nv.RECOMMEND_MAXX - T + 1                 # fits alone, not with the session's T clicks
    for off, ids, clicked, what in [(good_off, np.array([1, 2, 3, N, 5]), False, "session 3"),
                                    (good_off, np.array([1, -1, 3, 4, 5]), False, "session 0"),
                                    (np.array([0, 2, 1, 3, 5]), good_ids, False, "session 1"),
                                    (np.array([0, 1, 1, 1, nv.RECOMMEND_MAXX + 2]),
                                     np.zeros(nv.RECOMMEND_MAXX + 2, np.int32), False, "session 3"),
                                    (np.array([0, 0, long, long, long]), np.zeros(long, np.int32), True, "session 1"),
                                    (good_off[:-1], good_ids[:3], False, "offsets from 0")]:
        with pytest.raises(ValueError, match=what):
            model.recommend(bt, 5, off, ids, exclude_clicked=clicked)
    assert nv.LAUNCHES["count"] == before, "validation happens before any launch"
    model.recommend(bt, 5, np.array([0, 0, long, long, long]), np.zeros(long, np.int32))     # fine without clicks
    torch.cuda.synchronize()
    ps, p = model.ps, nv.ptr
    ws = torch.zeros(int(nv.lib().tcar_recommend_ws_bytes(B)), device=model.dev, dtype=torch.uint8)
    out_f, out_i = torch.zeros(8 * 300, device=model.dev), torch.zeros(8 * 300, device=model.dev, dtype=torch.int32)
    base = [p(out_f), p(out_f), p(model.a_ic), p(model.Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(model.cat_stats),
            None, None, None, T, B, N, ps.n_pad, 5, p(ws), p(out_i), p(out_f), None, nv.stream_ptr()]
    for at, v in [(15, 0), (15, nv.RECOMMEND_MAXK + 1), (12, nv.QROWS + 1), (14, N - 1), (8, p(out_i)), (16, None),
                  (7, None)]:
        a = list(base)
        a[at] = v
        assert nv.lib().tcar_recommend(*a) == -1                              # TCAR_ERR_ARG
    assert nv.lib().tcar_recommend_ws_bytes(nv.QROWS + 1) == -1


def test_recommend_after_a_pending_lookahead_update():
    """train_step(bt, next_bt) leaves the table-wide Adam pass running beside the next forward: recommend must see the
    updated tables, i.e. equal recommend after an explicit sync_updates()."""
    N, B, T = 3000, 128, 3
    outs = []
    for explicit in (False, True):
        model, _, mwdhm, _ = build(N)
        tb, _ = batch_for(model, N, B, T, 20, mwdhm, seed=2)
        nb, _ = batch_for(model, N, B, T, 20, mwdhm, seed=3)
        eb, _ = batch_for(model, N, 64, 5, 0, mwdhm, seed=4)
        model.train_step(tb, nb)
        if explicit:
            model.sync_updates()
        outs.append([x.clone() for x in model.recommend(eb, 50, exclude_clicked=True)])
        model.sync_updates()
    torch.cuda.synchronize()
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_recommend_split_end_to_end(tmp_path, monkeypatch):
    """main.py --recommend_k 20 on a synthetic split writes one parseable line per session; without exact ties at the
    label (checked here) HR / MRR / nDCG@20 equal test()'s Recall / MRR / nDCG@20."""
    from tcar_b200 import main as tmain, synth
    from tcar_b200.sampler import Sampler
    N, n_test = 1500, 150
    monkeypatch.chdir(tmp_path)
    root = str(tmp_path) + "/synth/TCAR-mid/Normal/"
    synth.write_dataset(root, N=N, n_train=700, n_test=n_test, fold=0)
    args = tmain.build_parser().parse_args(["--datapath", str(tmp_path) + "/", "--dataset", "synth/TCAR-mid/",
                                            "--foldnum", "0", "--epoch", "1", "--batch_size", "64",
                                            "--recommend_k", "20"])
    model = tmain.main(args)
    got, want = model.last_recommend_metrics, model.last_metrics
    load = lambda name: pickle.load(open(root + name, "rb"))
    item_dict = load("item_dict_0.txt")
    lines = open(tmp_path / "saved" / "recommend_0.txt").read().splitlines()
    assert len(lines) == n_test == got["sessions"]
    session_dict = load("session_dict_test_0.pkl")
    keys = set()
    for line in lines:
        key, *pairs = line.split()
        keys.add(key)
        assert len(pairs) == 20
        arts = [a.rsplit(":", 1)[0] for a in pairs]
        scores = [float(a.rsplit(":", 1)[1]) for a in pairs]
        assert all(a in {str(x) for x in item_dict} for a in arts) and len(set(arts)) == 20
        assert scores == sorted(scores, reverse=True)
    assert keys == {str(k) for k in session_dict}
    # no exact tie between a label and another item among the top 21 (the GPU's own fp32 scores)
    test = (load("len_dict_test0.pkl"), session_dict, load("session_time_dict_test0.pkl"))
    sampler = Sampler(*test, batch_size=64, verbose=False)
    while sampler.has_next():
        packed, B, T, _ = sampler.next_packed()
        bt = model.to_device(torch.from_numpy(packed).pin_memory(), B, T, 0)
        ids, sc = [x.cpu().numpy() for x in model.recommend(bt, 21)]
        labels = packed[7 * B * T + 2 * B: 7 * B * T + 3 * B]
        lab_sc, _, _, _ = model.rerank(bt, np.arange(B + 1, dtype=np.int32), labels.astype(np.int32), metrics=False)
        lab_sc = lab_sc.cpu().numpy()
        for b in range(B):
            assert not ((sc[b] == lab_sc[b]) & (ids[b] != labels[b])).any(), "fixture must have no exact label ties"
    for g, w in (("hr", "recall"), ("mrr", "mrr"), ("ndcg", "ndcg")):
        assert abs(got[g] - want[w]) <= 1e-12, (g, got[g], want[w])


def test_batches_of_different_sizes_back_to_back():
    """The workspace serves every batch size: a smaller batch between two calls on a larger one changes nothing."""
    N = 9000
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    big, _ = batch_for(model, N, 100, 3, 0, mwdhm, seed=5)
    small, _ = batch_for(model, N, 40, 2, 0, mwdhm, seed=6)
    a = [x.clone() for x in model.recommend(big, 30, exclude_clicked=True)]
    s = [x.clone() for x in model.recommend(small, 20)]
    b = model.recommend(big, 30, exclude_clicked=True)
    top, _, _ = model.eval_step(small)
    torch.cuda.synchronize()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(s[0], top) and torch.equal(s[1], model.top_scores[:40])
