"""Candidate re-ranking (tcar_rerank / Seq2SeqAttNN.rerank / test_impressions) against an fp64 reference built on the
oracle's forward(), and against the full-catalog evaluation it must agree with bit for bit.

Reference: scores are the oracle's softmax_input (model_combine.py:138) at the listed ids; the order is (score desc,
id asc, input position asc); label_rank = 1 + #(negatives > label) (util.py:14); auc counts tied negatives 1/2."""
import math
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import tcar_oracle as O  # noqa: E402
from test_gpu_parity import batch_for, build, oracle_inputs  # noqa: E402


def rerank_ref(S, labels, off, ids):
    """fp64 reference of tcar_rerank on the oracle's score matrix S [B,N]: (scores, ranked, rank, auc, n_neg,
    list_margin, label_margin).  list_margin: adjacent gaps of the sorted distinct scores of the list and the label
    exceed 2e-5 |score| (the margin_ok rule of the full-catalog tests); label_margin: the same for the label's gaps to
    its negatives only (what rank and auc depend on)."""
    sc, rk, ranks, aucs, nneg, lm, lab_m = [], [], [], [], [], [], []
    for b in range(len(off) - 1):
        c = ids[off[b]:off[b + 1]].astype(np.int64)
        s = S[b, c]
        sc.append(s)
        rk.append(c[np.lexsort((np.arange(len(c)), c, -s))])
        ls = S[b, labels[b]]
        sn = s[c != labels[b]]
        n = len(sn)
        ranks.append(1 + int((sn > ls).sum()))                          # brute-force pairwise counting
        aucs.append(((sn < ls).sum() + 0.5 * (sn == ls).sum()) / n if n else math.nan)
        nneg.append(n)
        u = np.unique(np.append(c, labels[b]))
        su = np.sort(S[b, u])
        scale = np.abs(su).max()
        lm.append(bool((np.diff(su) > 2e-5 * scale).all()))
        lab_m.append(bool((np.abs(sn - ls) > 2e-5 * scale).all()))
    return (np.concatenate(sc) if sc else np.zeros(0), np.concatenate(rk) if rk else np.zeros(0, np.int64),
            np.array(ranks), np.array(aucs), np.array(nneg), np.array(lm), np.array(lab_m))


def oracle_scores(model, content, mwdhm, batch):
    params, c64, m64 = oracle_inputs(model, content, mwdhm)
    with torch.no_grad():
        return O.forward(params, c64, m64, batch)["softmax_input"].numpy()


def make_lists(rs, N, lens, labels, dup=False):
    """CSR lists of the given lengths; every other list contains its label, `dup` repeats a few entries."""
    off = np.zeros(len(lens) + 1, dtype=np.int32)
    off[1:] = np.cumsum(lens)
    ids = rs.randint(0, N, int(off[-1])).astype(np.int32)
    for b, L in enumerate(lens):
        if L and b % 2 == 0:
            ids[off[b] + rs.randint(L)] = labels[b]
        if dup and L > 2:
            ids[off[b] + L - 1] = ids[off[b]]
    return off, ids


def host_order(scores, ids, off):
    """(score desc, id asc, position asc) of the GPU's own fp32 scores, per list."""
    out = []
    for b in range(len(off) - 1):
        s, c = scores[off[b]:off[b + 1]], ids[off[b]:off[b + 1]].astype(np.int64)
        out.append(c[np.lexsort((np.arange(len(c)), c, -s.astype(np.float64)))])
    return np.concatenate(out) if out else np.zeros(0, np.int64)


def lognormal_lens(N, B, seed):
    from tcar_b200 import synth
    return [len(v) for v in synth.make_impressions(N, B, seed=seed).values()]


@pytest.mark.parametrize("B,T,N,kind", [(1, 1, 300, "one"), (7, 3, 2000, "mixed"), (512, 20, 9000, "lognormal"),
                                        (64, 40, 70000, "maxl")])
def test_rerank_matches_fp64_reference(B, T, N, kind):
    from tcar_b200 import _native as nv
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=B + T)
    labels = batch["label"].numpy()
    rs = np.random.RandomState(B)
    lens = {"one": [1], "mixed": [0, 1, 2, 5, 37, 100, 300], "lognormal": lognormal_lens(N, B, 5),
            "maxl": [nv.RERANK_MAXL] + rs.randint(0, nv.RERANK_MAXL + 1, B - 1).tolist()}[kind]
    off, ids = make_lists(rs, N, lens, labels, dup=kind == "mixed")
    scores, ranked, rank, auc = model.rerank(bt, off, ids)
    again = [x.clone() for x in model.rerank(bt, off, ids)]
    torch.cuda.synchronize()
    for x, y in zip((scores, ranked, rank, auc), again):
        assert torch.equal(x, y) or (x.is_floating_point() and torch.equal(x.isnan(), y.isnan()) and
                                     torch.equal(x[~x.isnan()], y[~y.isnan()])), "second run must be bit-identical"
    S = oracle_scores(model, content, mwdhm, batch)
    r_sc, r_rk, r_rank, r_auc, r_nneg, lm, lab_m = rerank_ref(S, labels, off, ids)
    g_sc, g_rk = scores.cpu().numpy(), ranked.cpu().numpy()
    g_rank, g_auc = rank.cpu().numpy(), auc.cpu().numpy()
    np.testing.assert_allclose(g_sc, r_sc, rtol=1e-4, atol=1e-5)
    # the order is exactly (score desc, id asc, position asc) of the kernel's own scores on every list ...
    assert (g_rk == host_order(g_sc, ids, off)).all()
    # ... and the oracle's order wherever the oracle's scores are separated by more than the fp32 error
    el = np.repeat(lm, np.diff(off))
    assert (g_rk[el] == r_rk[el]).all()
    if kind != "maxl":                    # 2048 random scores nearly always hold some pair closer than 2e-5
        assert lm.mean() > 0.5, "fixture must be mostly margin-checked"
    assert lab_m.mean() > 0.8
    assert (g_rank == r_rank)[lab_m].all()
    ok = lab_m & (r_nneg > 0)
    np.testing.assert_allclose(g_auc[ok], r_auc[ok], rtol=0, atol=1e-6)
    assert np.isnan(g_auc[r_nneg == 0]).all()


def test_rerank_agrees_bit_for_bit_with_the_full_catalog_top20():
    """Re-ranking each query's eval_step top-20 (+ its label) reproduces the top-20 scores exactly, the top-20 order,
    and the rank eval_step counts whenever the label is inside its top-20."""
    from tcar_b200.sampler import impression_candidates
    N, B, T = 30000, 256, 4
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=21)
    # every other query's label is moved into its top-20 (at position b % 20); the labels do not change the top-20
    top0 = model.eval_step(bt)[0].cpu().numpy()
    labels = batch["label"].numpy().astype(np.int32)
    even = np.arange(0, B, 2)
    labels[even] = top0[even, even % 20]
    bt.label.copy_(torch.from_numpy(labels).to(model.dev))
    top, ngt, _ = [x.clone() for x in model.eval_step(bt)]
    top_sc = model.top_scores[:B].clone()
    top_np = top.cpu().numpy()
    assert (top_np == top0).all()
    arts = {b: top_np[b].tolist() for b in range(B)}
    off, ids = impression_candidates(list(range(B)), labels, arts, {i: i + 1 for i in range(N)})
    scores, ranked, rank, _ = model.rerank(bt, off, ids)
    torch.cuda.synchronize()
    scores, ranked, rank, ngt = scores.cpu(), ranked.cpu().numpy(), rank.cpu().numpy(), ngt.cpu().numpy()
    inside = np.array([labels[b] in top_np[b] for b in range(B)])
    assert inside.any() and (~inside).any()
    for b in range(B):
        lo = off[b]
        assert torch.equal(scores[lo:lo + 20], top_sc[b].cpu()), b
        assert (ranked[lo:lo + 20] == top_np[b]).all(), b
    assert (rank[inside] == ngt[inside] + 1).all()


def test_rerank_ties():
    """Duplicate item / content / publish-time rows score identically: the lower id comes first, the label wins ties
    in label_rank and a tied negative counts 1/2 in auc."""
    from tcar_b200.params import ParamStore
    N, B, T = 2000, 32, 3
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    p = model.ps.export()
    rs = np.random.RandomState(4)
    src = rs.choice(N // 2 - 1, 200, replace=False) * 2          # disjoint twin pairs (2k, 2k + 1)
    cont, mw = content.copy(), mwdhm.copy()
    for s_ in src:
        p["item"][s_ + 2] = p["item"][s_ + 1]
        cont[s_ + 2] = cont[s_ + 1]
        mw[s_ + 1] = mw[s_]
    model.ps = ParamStore(N, cont, mw, model.dev)
    model.ps.load(p)
    bt, batch = batch_for(model, N, B, T, 0, mw, seed=8)
    # session b: label = the higher id of a twin pair, list = [label, its twin, 10 other ids, the label again]
    labels = (src[:B] + 1).astype(np.int32)
    bt.label.copy_(torch.from_numpy(labels).to(model.dev))
    lists = [[int(labels[b]), int(src[b])] + [int(x) for x in rs.randint(0, N, 20) if x // 2 != src[b] // 2][:10] +
             [int(labels[b])] for b in range(B)]
    off = np.cumsum([0] + [len(x) for x in lists]).astype(np.int32)
    ids = np.concatenate(lists).astype(np.int32)
    scores, ranked, rank, auc = model.rerank(bt, off, ids)
    torch.cuda.synchronize()
    sc, rk, rank, auc = scores.cpu().numpy(), ranked.cpu().numpy(), rank.cpu().numpy(), auc.cpu().numpy()
    assert (rk == host_order(sc, ids, off)).all()
    for b in range(B):
        s, c, r = sc[off[b]:off[b + 1]], ids[off[b]:off[b + 1]], list(rk[off[b]:off[b + 1]])
        assert s[0] == s[1] and s[0] == s[-1], "twin rows must tie exactly"
        pos_src, pos_dst = r.index(src[b]), r.index(labels[b])
        assert pos_dst == pos_src + 1 and r[pos_dst + 1] == labels[b], "ties: lower id first, equal ids by position"
        sn = s[c != labels[b]]
        gt, eq = int((sn > s[0]).sum()), int((sn == s[0]).sum())
        assert eq >= 1
        assert rank[b] == 1 + gt, "the label wins ties"
        assert abs(auc[b] - (len(sn) - gt - eq + 0.5 * eq) / len(sn)) <= 1e-6


def test_rerank_input_checks():
    from tcar_b200 import _native as nv
    N, B, T = 500, 4, 2
    model, _, mwdhm, _ = build(N)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=1)
    good_off, good_ids = np.array([0, 2, 3, 3, 5]), np.array([1, 2, 3, 4, 5])
    before = nv.LAUNCHES["count"]
    for off, ids, what in [(good_off, np.array([1, 2, 3, N, 5]), "session 3"),
                           (np.array([0, 2, 1, 3, 5]), good_ids, "session 1"),
                           (np.array([0, 1, 1, 1, nv.RERANK_MAXL + 2]), np.zeros(nv.RERANK_MAXL + 2, np.int32),
                            "session 3"),
                           (good_off[:-1], good_ids[:3], "offsets from 0")]:
        with pytest.raises(ValueError, match=what):
            model.rerank(bt, off, ids)
    assert nv.LAUNCHES["count"] == before, "validation happens before any launch"
    ps, p = model.ps, nv.ptr
    d_off = torch.zeros(B + 1, device=model.dev, dtype=torch.int32)
    out_f, out_i = torch.zeros(8, device=model.dev), torch.zeros(8, device=model.dev, dtype=torch.int32)
    for Bc, max_len in [(B, nv.RERANK_MAXL + 1), (nv.QROWS + 1, 1), (-1, 1)]:
        rc = nv.lib().tcar_rerank(p(model.a_ic), p(model.Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(d_off),
                                  p(out_i), p(bt.label), Bc, N, max_len, p(out_f), p(out_i), p(out_i), p(out_f),
                                  nv.stream_ptr())
        assert rc == -1                                                     # TCAR_ERR_ARG


def test_rerank_after_a_pending_lookahead_update():
    """train_step(bt, next_bt) leaves the table-wide Adam pass running beside the next forward: rerank must see the
    updated tables, i.e. equal rerank after an explicit sync_updates()."""
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
        off, ids = make_lists(np.random.RandomState(0), N, [30] * 64, eb.label.cpu().numpy())
        outs.append([x.clone() for x in model.rerank(eb, off, ids)])
        model.sync_updates()
    torch.cuda.synchronize()
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_impression_eval_end_to_end(tmp_path):
    """main.py --impression_eval on a pickle-layout split: per-session ranks equal the fp64 reference on margin-checked
    sessions, the averages agree within 1e-3, and sessions without a negative are counted as skipped."""
    from tcar_b200 import main as tmain, synth
    from tcar_b200.sampler import Sampler, impression_candidates
    from tcar_b200.util import impression_metrics, impression_sums
    N, n_test = 1500, 150
    root = str(tmp_path) + "/synth/TCAR-mid/Normal/"
    synth.write_dataset(root, N=N, n_train=700, n_test=n_test, fold=0)
    impressions = synth.make_impressions(N, n_test)
    impressions[0] = ["x1", "x2"]                       # a session whose list holds no known article: skipped
    with open(root + "impressions.pkl", "wb") as f:
        pickle.dump(impressions, f)
    args = tmain.build_parser().parse_args(["--datapath", str(tmp_path) + "/", "--dataset", "synth/TCAR-mid/",
                                            "--foldnum", "0", "--epoch", "1", "--batch_size", "64",
                                            "--impression_path", root + "impressions.pkl", "--impression_eval"])
    model = tmain.main(args)
    got = model.last_impression_metrics
    # fp64 reference over the same split, session by session
    load = lambda name: pickle.load(open(root + name, "rb"))
    test = (load("len_dict_test0.pkl"), load("session_dict_test_0.pkl"), load("session_time_dict_test0.pkl"))
    item_dict, content, mw = load("item_dict_0.txt"), load("content_weight_0.txt"), load("publish_time_0.txt")[1]
    sampler = Sampler(*test, batch_size=64, verbose=False)
    sums, n_ok, n_all = np.zeros(6), 0, 0
    while sampler.has_next():
        keys = sampler.session_id_batches[sampler.batch_i]
        packed, B, T, Nn = sampler.next_packed()
        bt = model.to_device(torch.from_numpy(packed).pin_memory(), B, T, 0)
        batch = {k: torch.from_numpy(v) for k, v in synth.unpack(packed, B, T, 0).items()}
        labels = batch["label"].numpy()
        off, ids = impression_candidates(keys, labels, impressions, item_dict)
        _, _, rank, auc = model.rerank(bt, off, ids)
        S = oracle_scores(model, content, mw, batch)
        _, _, r_rank, r_auc, r_nneg, _, lab_m = rerank_ref(S, labels, off, ids)
        assert (rank.cpu().numpy() == r_rank)[lab_m].all()
        n_ok, n_all = n_ok + int(lab_m.sum()), n_all + B
        sums += impression_sums(r_rank, r_auc, r_nneg)
    want = impression_metrics(sums)
    assert n_all == n_test and n_ok >= 0.95 * n_all
    assert got["skipped"] == want["skipped"] >= 1 and got["sessions"] == want["sessions"] == n_test - want["skipped"]
    for k in ("auc", "mrr", "ndcg5", "ndcg10"):
        assert abs(got[k] - want[k]) <= 1e-3, (k, got[k], want[k])
